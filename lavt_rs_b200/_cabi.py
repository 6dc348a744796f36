"""ctypes binding of ``include/lavt_b200.h`` (the C-ABI of the sm_100a kernels).

The product path has NO CPU fallback: if the shared library is missing or the device is not a
B200, every call raises.  PyTorch tensors are used only as device-memory containers; the library
sees raw pointers and the current CUDA stream.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LAVT_LIB_PATH") or os.path.join(_PKG, "_lib", "liblavt_b200.so")   # LAVT_LIB_PATH: A/B runs of debug builds

ACT_NONE, ACT_GELU, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4


class WinGeom(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("B", "D", "H", "W", "wd", "wh", "ww", "sd", "sh", "sw",
                 "nwd", "nwh", "nww", "N", "Wd", "Wh", "Ww")]

    def rows(self) -> int:
        return self.B * self.nwd * self.nwh * self.nww * self.N

    def tokens(self) -> int:
        return self.B * self.D * self.H * self.W


class Epilogue(C.Structure):
    _fields_ = [
        ("cscale", C.c_void_p), ("bias", C.c_void_p),
        ("act", C.c_int32), ("ldm", C.c_int32),
        ("mul", C.c_void_p), ("resid", C.c_void_p),
        ("out_f32", C.c_void_p), ("out_bf16", C.c_void_p),
        ("ldo", C.c_int32), ("mul_act", C.c_int32),
        ("win", C.POINTER(WinGeom)),
        ("rscale", C.c_void_p), ("rscale_rows", C.c_int32), ("pre_mode", C.c_int32),
        ("out_pre", C.c_void_p),
    ]


class LavtError(RuntimeError):
    pass


_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load the library (once). Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LavtError(
            f"{LIB_PATH} not found: build it with `python -m lavt_rs_b200.build` "
            "(the B200 path has no CPU / PyTorch fallback)")
    l = C.CDLL(LIB_PATH)
    l.lavt_last_error.restype = C.c_char_p
    _declare(l)
    if l.lavt_abi_version() != ABI_VERSION:
        raise LavtError("liblavt_b200.so ABI version mismatch; rebuild")
    _lib = l
    return l


ABI_VERSION = 4

_i32, _i64, _f32, _vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p
_EP = C.POINTER(Epilogue)
_WG = C.POINTER(WinGeom)

# name -> argtypes; every function returns int status.  Kept in the order of include/lavt_b200.h.
SIGNATURES = {
    "lavt_check_device": [],
    "lavt_gemm_bf16": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _EP, _vp],
    "lavt_gemm_bf16_smallm": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _EP, _vp, _i64, _vp],
    "lavt_conv3x3_bf16": [_vp, _i64, _i32, _i32, _i32, _i32, _vp, _i32, _EP, _vp],
    "lavt_conv3d_bf16": [_vp, _i64, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _EP, _vp],
    "lavt_layernorm_rows": [_vp, _i64, _i64, _i32, _vp, _vp, _f32, _vp, _vp, _vp],
    "lavt_layernorm_window_gather": [_vp, _i32, _WG, _vp, _vp, _f32, _vp, _vp],
    "lavt_patch_merge_layernorm": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _f32, _vp, _vp],
    "lavt_patch_embed_im2col": [_vp, _i64, _i64, _i64, _i32, _i32, _i32, _i32, _vp, _vp],
    "lavt_window_attention": [_vp, _vp, _i32, _i32, _WG, _vp, _vp],
    "lavt_window_attention_lse": [_vp, _vp, _i32, _i32, _WG, _vp, _vp, _vp],
    "lavt_instnorm_stats": [_vp, _i32, _i64, _i32, _f32, _vp, _vp, _vp],
    "lavt_pwam_kv": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_lang_project": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_lang_project_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_pwam_attend": [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _vp],
    "lavt_pwam_mul_norm": [_vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_instnorm_sum2": [_vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_bert_embed": [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_bert_attention": [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_rows_to_channels_first": [_vp, _vp, _i32, _i32, _i32, _vp],
    "lavt_split3_bf16": [_vp, _i64, _vp, _i64, _i32, _vp],
    "lavt_bert_attention_f32": [_vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_upsample_concat": [_vp, _i32, _i32, _i32, _vp, _i32, _vp, _i32, _i32, _i32, _vp],
    "lavt_upconv_blend": [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp],
    "lavt_conv1x1_logits": [_vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "lavt_upsample_logits": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_nhwc_to_nchw": [_vp, _vp, _i32, _i32, _i32, _vp],
    "lavt_nchw_to_nhwc_bf16": [_vp, _vp, _i32, _i32, _i32, _vp],
    # ---- backward pass ----
    "lavt_gemm_bf16_splitk": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _i64, _i32, _vp],
    "lavt_gemm_bf16_wgrad": [_vp, _i64, _vp, _i64, _i64, _i32, _i32, _vp, _i64, _vp, _i64, _i32, _vp],
    "lavt_conv3x3_wgrad": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _i32, _vp],
    "lavt_conv3d_wgrad": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _i32, _vp],
    "lavt_transpose_bf16": [_vp, _i64, _vp, _i64, _i64, _i32, _vp],
    "lavt_colsum_accumulate": [_vp, _i32, _i64, _i64, _i32, _vp, _vp],
    "lavt_cast_rows_bf16": [_vp, _i64, _i64, _i32, _WG, _vp, _vp],
    "lavt_cast_rows_scaled_bf16": [_vp, _i64, _i64, _i32, _WG, _vp, _i32, _vp, _vp],
    "lavt_cast_rows_colsum_bf16": [_vp, _i64, _i64, _i32, _WG, _vp, _i32, _vp, _vp, _vp],
    "lavt_gelu_fwd": [_vp, _vp, _i64, _vp],
    "lavt_gelu_bwd": [_vp, _vp, _vp, _i64, _vp],
    "lavt_layernorm_rows_bwd": [_vp, _i64, _i64, _i32, _vp, _i64, _vp, _f32, _vp, _vp, _vp, _vp, _vp],
    "lavt_layernorm_window_gather_bwd": [_vp, _i32, _WG, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _vp],
    "lavt_patch_merge_layernorm_bwd": [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp],
    "lavt_window_attention_bwd": [_vp, _vp, _vp, _vp, _i32, _i32, _WG, _vp, _vp, _vp, _vp, _i64, _vp],
    "lavt_pwam_attend_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _i32, _vp],
    "lavt_pwam_mul_norm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_instnorm_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_pwam_kv_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_gate_elementwise": [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp],
    "lavt_bn_relu_apply": [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "lavt_bn_relu_bwd_reduce": [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "lavt_bn_relu_bwd_apply": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp],
    "lavt_nhwc_pad_transpose": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_instnorm_bwd_reduce": [_vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_upsample_concat_bwd": [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_conv1x1_logits_bwd": [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp],
    "lavt_upsample_logits_bwd": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_cross_entropy": [_vp, _vp, _f32, _f32, _vp, _vp, _f32, _i32, _i32, _i32, _i32, _vp],
    "lavt_normalize_u8": [_vp, _vp, _i32, _i32, _i32, _vp, _vp, _vp],
    "lavt_logits_to_mask": [_vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_gacd_fuse": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i64, _i32, _vp],
    "lavt_adamw_step": [_vp, _vp, _i32, _i32, _f32, C.c_double, C.c_double, _f32, _f32, _vp],
    "lavt_bcam_words": [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp],
    "lavt_efn_sentence_bias": [_vp, _vp, _vp, _i64, _vp, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_efn_word_attend": [_vp, _i64, _vp, _vp, _i64, _vp, _i32, _i64, _i32, _i32, _vp],
    "lavt_efn_norm_pool": [_vp, _vp, _vp, _i32, _i64, _i32, _i32, _i64, _i32, _vp],
    "lavt_efn_norm_upsample": [_vp, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _vp],
    "lavt_bcam_softmax_rows": [_vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32, _vp],
    "lavt_bcam_transpose_pad": [_vp, _i64, _vp, _i64, _i32, _i64, _i32, _vp],
    "lavt_gemm_f32_ref": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _EP, _vp],
    "lavt_window_attention_f32_ref": [_vp, _vp, _i32, _i32, _WG, _vp, _vp],
    "lavt_layernorm_window_gather_f32": [_vp, _i32, _WG, _vp, _vp, _f32, _vp, _vp],
    "lavt_rows_affine_act": [_vp, _i32, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i32, _vp, _vp, _i64, _i64, _i32, _vp],
    "lavt_avgpool2_nhwc": [_vp, _i64, _vp, _i64, _i32, _i32, _i32, _i32, _vp],
    "lavt_append_coords": [_vp, _i64, _vp, _i32, _i32, _i32, _i32, _vp],
    "lavt_rows_add_table": [_vp, _i32, _i64, _vp, _i64, _vp, _vp, _i64, _i64, _i32, _vp],
    "lavt_mha_small": [_vp, _i64, _vp, _i64, _vp, _i64, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _vp],
    "lavt_gate_transpose": [_vp, _i64, _vp, _i64, _vp, _i32, _i32, _i32, _vp],
}
EXPORTS = ["lavt_last_error", "lavt_abi_version", "lavt_instnorm_workspace_floats", "lavt_set_attention_impl", "lavt_set_attention_bwd_impl",
           "lavt_gemm_splitk_workspace_floats", "lavt_conv3x3_wgrad_workspace_floats", "lavt_gacd_workspace_floats", "lavt_conv3d_wgrad_workspace_floats", "lavt_adamw_chunk_elems", "lavt_window_attention_has_lse",
           "lavt_window_attention_bwd_kernel", "lavt_window_attention_bwd_workspace_floats",
           *SIGNATURES.keys()]


def _declare(l: C.CDLL) -> None:
    l.lavt_abi_version.restype = C.c_int
    l.lavt_instnorm_workspace_floats.argtypes = [_i32, _i64, _i32]
    l.lavt_instnorm_workspace_floats.restype = C.c_int64
    l.lavt_gemm_splitk_workspace_floats.argtypes = [_i32, _i32, _i32]
    l.lavt_gemm_splitk_workspace_floats.restype = C.c_int64
    l.lavt_window_attention_has_lse.argtypes = [_WG, _i32, _i32]
    l.lavt_window_attention_has_lse.restype = C.c_int
    l.lavt_window_attention_bwd_kernel.argtypes = [_WG, _i32, _i32, _i32]
    l.lavt_window_attention_bwd_kernel.restype = C.c_int
    l.lavt_window_attention_bwd_workspace_floats.argtypes = [_WG, _i32, _i32]
    l.lavt_window_attention_bwd_workspace_floats.restype = C.c_int64
    l.lavt_conv3x3_wgrad_workspace_floats.argtypes = [_i32, _i32, _i32, _i32, _i32]
    l.lavt_conv3x3_wgrad_workspace_floats.restype = C.c_int64
    l.lavt_conv3d_wgrad_workspace_floats.argtypes = [_i32, _i32, _i32, _i32, _i32, _i32]
    l.lavt_conv3d_wgrad_workspace_floats.restype = C.c_int64
    l.lavt_gacd_workspace_floats.argtypes = [_i32, _i64, _i32]
    l.lavt_gacd_workspace_floats.restype = C.c_int64
    l.lavt_adamw_chunk_elems.argtypes = []
    l.lavt_adamw_chunk_elems.restype = C.c_int
    l.lavt_set_attention_impl.argtypes = [_i32]
    l.lavt_set_attention_impl.restype = C.c_int
    l.lavt_set_attention_bwd_impl.argtypes = [_i32]
    l.lavt_set_attention_bwd_impl.restype = C.c_int
    for name, argtypes in SIGNATURES.items():
        fn = getattr(l, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().lavt_last_error().decode(errors="replace")
        raise LavtError(f"{what} failed (code {rc}): {msg}")


_RAW_STREAM = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr() -> int:
    """cudaStream_t of torch's current stream (the raw getter skips the Stream object ``torch.cuda.current_stream()`` builds on every call)."""
    if _RAW_STREAM is not None:
        return _RAW_STREAM(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _req(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise LavtError(f"{name} must be a CUDA tensor (no CPU fallback)")
    if t.dtype != dtype:
        raise LavtError(f"{name} must be {dtype}, got {t.dtype}")
    if t.stride(-1) != 1:
        raise LavtError(f"{name} must be contiguous in its last dimension")


def make_epilogue(*, cscale=None, bias=None, act=ACT_NONE, mul=None, resid=None,
                  out_f32=None, out_bf16=None, ldo=None, win: Optional[WinGeom] = None, rscale=None, rscale_rows: int = 0,
                  mul_act=ACT_NONE, out_pre=None, pre_mode: int = 0) -> Epilogue:
    """``mul_act=ACT_GELU``: the result is multiplied by GELU'(mul) instead of mul; ``out_pre`` (bf16): the value before the activation,
    or with ``pre_mode=1`` (act = GELU) the derivative GELU'(pre)."""
    e = Epilogue()
    for name, t in (("cscale", cscale), ("bias", bias), ("resid", resid), ("out_f32", out_f32)):
        if t is not None:
            _req(t, torch.float32, name)
    for name, t in (("mul", mul), ("out_bf16", out_bf16), ("out_pre", out_pre)):
        if t is not None:
            _req(t, torch.bfloat16, name)
    e.cscale, e.bias = ptr(cscale), ptr(bias)
    e.act = act
    e.mul = ptr(mul)
    e.ldm = mul.stride(-2) if mul is not None else 0
    e.mul_act = mul_act
    e.out_pre = ptr(out_pre)
    e.pre_mode = int(pre_mode)
    e.resid = ptr(resid)
    e.out_f32, e.out_bf16 = ptr(out_f32), ptr(out_bf16)
    out = out_f32 if out_f32 is not None else out_bf16
    if out is None:
        raise LavtError("epilogue needs out_f32 or out_bf16")
    e.ldo = int(ldo if ldo is not None else out.stride(-2))
    for t in (resid, out_f32, out_bf16, out_pre):
        if t is not None and t.stride(-2) != e.ldo:
            raise LavtError("resid / out_f32 / out_bf16 / out_pre must share one row pitch")
    e.win = C.pointer(win) if win is not None else None
    if rscale is not None:
        _req(rscale, torch.float32, "rscale")
        if rscale_rows <= 0:
            raise LavtError("rscale needs rscale_rows > 0")
        e.rscale, e.rscale_rows = rscale.data_ptr(), int(rscale_rows)
    return e


class KernelTimer:
    """Optional CUDA-event timing of individual launches (bench.py roofline leg). Disabled by default."""

    def __init__(self):
        self.enabled = False
        self.records = []   # (family, flops, bytes, start_event, end_event)

    def begin(self):
        if not self.enabled:
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def end(self, start, family: str, flops: float, nbytes: float, tag: str = ""):
        if start is None:
            return
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        self.records.append((family, flops, nbytes, start, ev, tag))

    def by_tag(self):
        torch.cuda.synchronize()
        out = {}
        for fam, fl, nb, s, e, tag in self.records:
            d = out.setdefault((fam, tag), {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0})
            d["launches"] += 1
            d["ms"] += s.elapsed_time(e)
            d["flops"] += fl
            d["bytes"] += nb
        return out

    def summary(self, peak_tflops: float = 0.0, peak_gbs: float = 0.0):
        """Per kernel family: launches, total ms, algorithmic FLOPs / bytes and (given the two peaks) the sum over
        launches of the roofline-ideal time max(flops / peak_tflops, bytes / peak_gbs)."""
        torch.cuda.synchronize()
        out = {}
        for fam, fl, nb, s, e, _tag in self.records:
            d = out.setdefault(fam, {"launches": 0, "ms": 0.0, "flops": 0.0, "bytes": 0.0, "ideal_ms": 0.0})
            d["launches"] += 1
            d["ms"] += s.elapsed_time(e)
            d["flops"] += fl
            d["bytes"] += nb
            if peak_tflops > 0 and peak_gbs > 0:
                d["ideal_ms"] += max(fl / (peak_tflops * 1e12), nb / (peak_gbs * 1e9)) * 1e3
        return out


TIMER = KernelTimer()


def gemm_bf16(a: torch.Tensor, w: torch.Tensor, **epi) -> None:
    """out = epilogue(a @ w.T); a [M,K] bf16, w [N,K] bf16 (nn.Linear layout)."""
    _req(a, torch.bfloat16, "a")
    _req(w, torch.bfloat16, "w")
    M, K = a.shape
    N, K2 = w.shape
    if K != K2:
        raise LavtError(f"gemm: K mismatch {K} vs {K2}")
    e = make_epilogue(**epi)
    t0 = TIMER.begin()
    check(lib().lavt_gemm_bf16(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M, N, K,
                               C.byref(e), stream_ptr()), "lavt_gemm_bf16")
    if t0 is not None:
        nbytes = 2.0 * (M * K + N * K) + M * N * ((4.0 if e.out_f32 else 0.0) + (2.0 if e.out_bf16 else 0.0)
                                                   + (4.0 if e.resid else 0.0) + (2.0 if e.mul else 0.0))
        TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * M * N * K, nbytes, f"M{M} N{N} K{K} act{e.act}")


def gemm_bf16_smallm(a: torch.Tensor, w: torch.Tensor, workspace: torch.Tensor, **epi) -> None:
    """gemm_bf16 for a few rows (the text encoder: M = clips x words): split-K launch that fills the GPU + one reduce / epilogue kernel.
    ``workspace`` fp32 with at least splitk_workspace_floats(M, N, K) elements; epilogue: cscale, bias, act (none / GELU), resid, out_f32, out_bf16."""
    _req(a, torch.bfloat16, "a")
    _req(w, torch.bfloat16, "w")
    M, K = a.shape
    N, K2 = w.shape
    if K != K2:
        raise LavtError(f"gemm: K mismatch {K} vs {K2}")
    e = make_epilogue(**epi)
    check(lib().lavt_gemm_bf16_smallm(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M, N, K, C.byref(e),
                                      _c(workspace, torch.float32, "workspace").data_ptr(), workspace.numel(), stream_ptr()),
          "lavt_gemm_bf16_smallm")


def conv3x3_bf16(x_nhwc: torch.Tensor, w_taps: torch.Tensor, **epi) -> None:
    """x [n_img,H,W,Cin] bf16 NHWC; w_taps [Cout, 9*Cin] bf16 (tap-major: (ky*3+kx)*Cin+ci)."""
    _req(x_nhwc, torch.bfloat16, "x")
    _req(w_taps, torch.bfloat16, "w_taps")
    n_img, H, W, Cin = x_nhwc.shape
    if not x_nhwc.is_contiguous():
        raise LavtError("conv: x must be contiguous NHWC")
    Cout = w_taps.shape[0]
    e = make_epilogue(**epi)
    t0 = TIMER.begin()
    check(lib().lavt_conv3x3_bf16(x_nhwc.data_ptr(), Cin, n_img, H, W, Cin, w_taps.data_ptr(), Cout,
                                  C.byref(e), stream_ptr()), "lavt_conv3x3_bf16")
    npix = n_img * H * W
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * npix * Cout * 9 * Cin, 2.0 * (npix * Cin + Cout * 9 * Cin + npix * Cout),
              f"conv {n_img}x{H}x{W} Cin{Cin} Cout{Cout}")


def conv3d_bf16(x_ndhwc: torch.Tensor, w_taps: torch.Tensor, **epi) -> None:
    """x [n_clip,D,H,W,Cin] bf16 NDHWC; w_taps [Cout, 27*Cin] bf16 (tap-major: ((kz*3+ky)*3+kx)*Cin+ci)."""
    _req(x_ndhwc, torch.bfloat16, "x")
    _req(w_taps, torch.bfloat16, "w_taps")
    n_clip, D, H, W, Cin = x_ndhwc.shape
    if not x_ndhwc.is_contiguous():
        raise LavtError("conv3d: x must be contiguous NDHWC")
    Cout = w_taps.shape[0]
    e = make_epilogue(**epi)
    t0 = TIMER.begin()
    check(lib().lavt_conv3d_bf16(x_ndhwc.data_ptr(), Cin, n_clip, D, H, W, Cin, w_taps.data_ptr(), Cout,
                                 C.byref(e), stream_ptr()), "lavt_conv3d_bf16")
    npos = n_clip * D * H * W
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * npos * Cout * 27 * Cin, 2.0 * (npos * Cin + Cout * 27 * Cin + npos * Cout),
              f"conv3d {n_clip}x{D}x{H}x{W} Cin{Cin} Cout{Cout}")


# ------------------------------------------------------------------------------------------------
# row kernels
# ------------------------------------------------------------------------------------------------
def _c(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    _req(t, dtype, name)
    if not t.is_contiguous():
        raise LavtError(f"{name} must be contiguous")
    return t


def layernorm_rows(x: torch.Tensor, gamma, beta, *, out_bf16=None, out_f32=None, eps: float = 1e-5) -> None:
    """x fp32 [M, C] (row pitch x.stride(0))."""
    _req(x, torch.float32, "x")
    M, Cn = x.shape
    for t, dt, nm in ((out_bf16, torch.bfloat16, "out_bf16"), (out_f32, torch.float32, "out_f32")):
        if t is not None:
            _c(t, dt, nm)
    check(lib().lavt_layernorm_rows(x.data_ptr(), x.stride(0), M, Cn, _c(gamma, torch.float32, "gamma").data_ptr(),
                                    _c(beta, torch.float32, "beta").data_ptr(), eps, ptr(out_bf16), ptr(out_f32),
                                    stream_ptr()), "lavt_layernorm_rows")


def layernorm_window_gather(x: torch.Tensor, geom: WinGeom, gamma, beta, out_bf16: torch.Tensor, eps: float = 1e-5) -> None:
    """x fp32 [(B*D*H*W), C] contiguous -> out bf16 [geom.rows(), C] in window order."""
    _c(x, torch.float32, "x")
    Cn = x.shape[-1]
    if x.numel() != geom.tokens() * Cn or out_bf16.numel() != geom.rows() * Cn:
        raise LavtError("window gather: tensor sizes do not match the geometry")
    check(lib().lavt_layernorm_window_gather(x.data_ptr(), Cn, C.byref(geom), _c(gamma, torch.float32, "gamma").data_ptr(),
                                             _c(beta, torch.float32, "beta").data_ptr(), eps,
                                             _c(out_bf16, torch.bfloat16, "out").data_ptr(), stream_ptr()),
          "lavt_layernorm_window_gather")


def patch_merge_layernorm(x: torch.Tensor, B, D, H, W, gamma, beta, out_bf16: torch.Tensor, eps: float = 1e-5) -> None:
    _c(x, torch.float32, "x")
    Cn = x.shape[-1]
    check(lib().lavt_patch_merge_layernorm(x.data_ptr(), B, D, H, W, Cn, _c(gamma, torch.float32, "gamma").data_ptr(),
                                           _c(beta, torch.float32, "beta").data_ptr(), eps,
                                           _c(out_bf16, torch.bfloat16, "out").data_ptr(), stream_ptr()),
          "lavt_patch_merge_layernorm")


def patch_embed_im2col(x: torch.Tensor, out_bf16: torch.Tensor) -> None:
    """x fp32 (B,3,T,H,W), any batch/channel/time strides as long as each (H,W) plane is contiguous."""
    _req(x, torch.float32, "x")
    B, Cin, T, H, W = x.shape
    if Cin != 3:
        raise LavtError("patch embed expects 3 input channels")
    if x.stride(3) != W:
        raise LavtError("patch embed: image planes must be contiguous")
    check(lib().lavt_patch_embed_im2col(x.data_ptr(), x.stride(0), x.stride(1), x.stride(2), B, T, H, W,
                                        _c(out_bf16, torch.bfloat16, "out").data_ptr(), stream_ptr()),
          "lavt_patch_embed_im2col")


def set_attention_impl(impl: str) -> str:
    """'auto' (attn_tc3.cu for full 7 x 7 / 12 x 12 windows, the chunked one-pass tcgen05 kernel attn_tc2.cu for every other window of
    16+ tokens, the mma.sync kernel for smaller ones), 'tc2' (attn_tc2.cu wherever it applies) or 'tc3' (the same as auto); returns the
    previous setting."""
    codes = {"auto": 0, "tc2": 3, "tc3": 4}
    if impl not in codes:
        raise LavtError(f"attention impl must be one of {sorted(codes)}, not {impl!r}")
    prev = lib().lavt_set_attention_impl(codes[impl])
    return {v: k for k, v in codes.items()}.get(prev, "auto")


ATTN_BWD_IMPLS = ("auto", "mma", "tc", "tc2")
ATTN_BWD_KERNELS = {0: None, 1: "mma", 2: "tc", 3: "tc2"}


def set_attention_bwd_impl(impl: str) -> str:
    """'auto' / 'tc' (tcgen05 kernel attn_bwd_tc.cu for 7 x 7 windows, else the mma.sync kernel where the window fits its shared
    memory, else the tcgen05 kernel attn_bwd_tc2.cu), 'mma' (mma.sync kernel only) or 'tc2' (attn_bwd_tc2.cu wherever it applies, else
    as auto); returns the previous setting."""
    if impl not in ATTN_BWD_IMPLS:
        raise LavtError(f"attention backward impl must be one of {list(ATTN_BWD_IMPLS)}, not {impl!r}")
    prev = lib().lavt_set_attention_bwd_impl(ATTN_BWD_IMPLS.index(impl))
    return ATTN_BWD_IMPLS[prev] if 0 <= prev < len(ATTN_BWD_IMPLS) else "auto"


def window_attention_bwd_kernel(table_t: torch.Tensor, geom: WinGeom, has_lse: bool = True) -> Optional[str]:
    """The kernel window_attention_bwd runs for this geometry under the current selection: 'mma', 'tc', 'tc2', or None (no kernel)."""
    nH, L = table_t.shape
    return ATTN_BWD_KERNELS[int(lib().lavt_window_attention_bwd_kernel(C.byref(geom), L, nH, 1 if has_lse else 0))]


def window_attention_bwd_workspace_floats(table_t: torch.Tensor, geom: WinGeom) -> int:
    """fp32 elements of the workspace window_attention_bwd needs for this geometry (with lse); 0 for most windows."""
    nH, L = table_t.shape
    return int(lib().lavt_window_attention_bwd_workspace_floats(C.byref(geom), L, nH))


def window_attention_has_lse(table_t: torch.Tensor, geom: WinGeom) -> bool:
    """True if window_attention can also write the per-row log-sum-exp for this geometry (tcgen05 kernels: windows of 16+ tokens)."""
    nH, L = table_t.shape
    return bool(lib().lavt_window_attention_has_lse(C.byref(geom), L, nH))


def window_attention(qkv: torch.Tensor, table_t: torch.Tensor, geom: WinGeom, out_bf16: torch.Tensor, lse: Optional[torch.Tensor] = None) -> None:
    """table_t: relative_position_bias_table transposed to [nH, L] fp32; lse: optional fp32 [rows, nH] row statistics (training)."""
    _c(qkv, torch.bfloat16, "qkv")
    _c(table_t, torch.float32, "table_t")
    nH, L = table_t.shape
    t0 = TIMER.begin()
    if lse is None:
        check(lib().lavt_window_attention(qkv.data_ptr(), table_t.data_ptr(), L, nH, C.byref(geom),
                                          _c(out_bf16, torch.bfloat16, "out").data_ptr(), stream_ptr()),
              "lavt_window_attention")
    else:
        check(lib().lavt_window_attention_lse(qkv.data_ptr(), table_t.data_ptr(), L, nH, C.byref(geom),
                                              _c(out_bf16, torch.bfloat16, "out").data_ptr(), _c(lse, torch.float32, "lse").data_ptr(),
                                              stream_ptr()), "lavt_window_attention_lse")
    rows = geom.rows()
    TIMER.end(t0, "window_attn_kernel", 4.0 * rows * geom.N * nH * 32, 2.0 * rows * nH * 32 * 4,
              f"rows{rows} N{geom.N} nH{nH} shift{geom.sh}")


def instnorm_workspace_floats(B: int, n: int, Cn: int) -> int:
    return int(lib().lavt_instnorm_workspace_floats(B, n, Cn))


def instnorm_stats(x: torch.Tensor, stats: torch.Tensor, workspace: torch.Tensor, eps: float = 1e-5) -> None:
    """x fp32 [B,n,C] -> stats fp32 [B,2,C] (mean, rstd)."""
    _c(x, torch.float32, "x")
    B, n, Cn = x.shape
    if workspace.numel() < instnorm_workspace_floats(B, n, Cn):
        raise LavtError("instnorm_stats: workspace too small")
    check(lib().lavt_instnorm_stats(x.data_ptr(), B, n, Cn, eps, _c(stats, torch.float32, "stats").data_ptr(),
                                    _c(workspace, torch.float32, "workspace").data_ptr(), stream_ptr()),
          "lavt_instnorm_stats")


def pwam_kv(l, mask, wk, bk, wv, bv, k, v) -> None:
    """l fp32 [B,Lin,Nl]; mask fp32 [B,Nl]; wk/wv fp32 [C,Lin]; k,v fp32 [B,Nl,C]."""
    B, Lin, Nl = l.shape
    Cn = wk.shape[0]
    for t, nm in ((l, "l"), (mask, "mask"), (wk, "wk"), (bk, "bk"), (wv, "wv"), (bv, "bv"), (k, "k"), (v, "v")):
        _c(t, torch.float32, nm)
    check(lib().lavt_pwam_kv(l.data_ptr(), mask.data_ptr(), wk.data_ptr(), bk.data_ptr(), wv.data_ptr(), bv.data_ptr(),
                             k.data_ptr(), v.data_ptr(), B, Nl, Lin, Cn, stream_ptr()), "lavt_pwam_kv")


def lang_project(l, mask, w0, b0, w2, b2, stats) -> None:
    """--fuse simple: stats fp32 [B,2,C] = (-LangProject(l, mask), 1); l fp32 [B,Lin,Nl], mask fp32 [B,Nl]."""
    B, Lin, Nl = l.shape
    Cn = w0.shape[0]
    for t, nm in ((l, "l"), (mask, "mask"), (w0, "w0"), (b0, "b0"), (w2, "w2"), (b2, "b2"), (stats, "stats")):
        _c(t, torch.float32, nm)
    check(lib().lavt_lang_project(l.data_ptr(), mask.data_ptr(), w0.data_ptr(), b0.data_ptr(), w2.data_ptr(), b2.data_ptr(),
                                  stats.data_ptr(), B, Nl, Lin, Cn, stream_ptr()), "lavt_lang_project")


def lang_project_bwd(l, mask, w0, b0, w2, ds, dw0, db0, dw2, db2, dl, workspace) -> None:
    """Adjoint of lang_project: ds fp32 [B,C]; dw0 / db0 / dw2 / db2 / dl accumulate (None = not needed)."""
    B, Lin, Nl = l.shape
    Cn = w0.shape[0]
    if workspace.numel() < B * (2 * Cn + 2 * Lin):
        raise LavtError("lang_project_bwd: workspace too small")
    check(lib().lavt_lang_project_bwd(_c(l, torch.float32, "l").data_ptr(), _c(mask, torch.float32, "mask").data_ptr(),
                                      _c(w0, torch.float32, "w0").data_ptr(), _c(b0, torch.float32, "b0").data_ptr(),
                                      _c(w2, torch.float32, "w2").data_ptr(), _c(ds, torch.float32, "ds").data_ptr(), ptr(dw0), ptr(db0),
                                      ptr(dw2), ptr(db2), ptr(dl), _c(workspace, torch.float32, "workspace").data_ptr(), B, Nl, Lin, Cn,
                                      stream_ptr()), "lavt_lang_project_bwd")


def pwam_attend(qpre, stats, k, v, mask, out, heads: int) -> None:
    _c(qpre, torch.float32, "qpre")
    B, n, Cn = qpre.shape
    Nl = k.shape[1]
    check(lib().lavt_pwam_attend(qpre.data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                 _c(k, torch.float32, "k").data_ptr(), _c(v, torch.float32, "v").data_ptr(),
                                 _c(mask, torch.float32, "mask").data_ptr(), _c(out, torch.bfloat16, "out").data_ptr(),
                                 B, n, Cn, Nl, heads, stream_ptr()), "lavt_pwam_attend")


def pwam_mul_norm(vis, lang, stats, out) -> None:
    _c(vis, torch.bfloat16, "vis")
    B, n, Cn = vis.shape
    check(lib().lavt_pwam_mul_norm(vis.data_ptr(), _c(lang, torch.float32, "lang").data_ptr(),
                                   _c(stats, torch.float32, "stats").data_ptr(), _c(out, torch.bfloat16, "out").data_ptr(),
                                   B, n, Cn, stream_ptr()), "lavt_pwam_mul_norm")


def instnorm_sum2(a, stats_a, b, stats_b, out) -> None:
    """out = IN(a) + IN(b); a, b, out fp32 [B,n,C]; stats fp32 [B,2,C] (mean, rstd)."""
    B, n, Cn = a.shape
    check(lib().lavt_instnorm_sum2(_c(a, torch.float32, "a").data_ptr(), _c(stats_a, torch.float32, "stats_a").data_ptr(),
                                   _c(b, torch.float32, "b").data_ptr(), _c(stats_b, torch.float32, "stats_b").data_ptr(),
                                   _c(out, torch.float32, "out").data_ptr(), B, n, Cn, stream_ptr()), "lavt_instnorm_sum2")


def bert_embed(ids, word, pos, type0, out) -> None:
    """ids int64 [B,Nl]; word [V,H], pos [P,H], type0 [H] fp32 -> out fp32 [B*Nl, H]."""
    if ids.dtype != torch.int64 or not ids.is_cuda or not ids.is_contiguous():
        raise LavtError("bert_embed: ids must be a contiguous CUDA int64 tensor")
    B, Nl = ids.shape
    V, H = word.shape
    if Nl > pos.shape[0]:
        raise LavtError("bert_embed: sentence longer than the position table")
    check(lib().lavt_bert_embed(ids.data_ptr(), _c(word, torch.float32, "word").data_ptr(), _c(pos, torch.float32, "pos").data_ptr(),
                                _c(type0, torch.float32, "type0").data_ptr(), _c(out, torch.float32, "out").data_ptr(), B, Nl, H, V,
                                stream_ptr()), "lavt_bert_embed")


def bert_attention(qkv, mask, out, heads: int) -> None:
    """qkv bf16 [B*Nl, 3H]; mask fp32 [B,Nl]; out bf16 [B*Nl, H]."""
    B, Nl = mask.shape
    H = out.shape[1]
    check(lib().lavt_bert_attention(_c(qkv, torch.bfloat16, "qkv").data_ptr(), _c(mask, torch.float32, "mask").data_ptr(),
                                    _c(out, torch.bfloat16, "out").data_ptr(), B, Nl, H, heads, stream_ptr()), "lavt_bert_attention")


def rows_to_channels_first(x, out) -> None:
    """x fp32 [B,Nl,C] -> out fp32 [B,C,Nl]."""
    B, Nl, Cn = x.shape
    check(lib().lavt_rows_to_channels_first(_c(x, torch.float32, "x").data_ptr(), _c(out, torch.float32, "out").data_ptr(), B, Nl, Cn,
                                            stream_ptr()), "lavt_rows_to_channels_first")


def upsample_concat(prev, skip, out) -> None:
    """prev bf16 [n,ph,pw,C1], skip bf16 [n,H,W,C2] -> out bf16 [n,H,W,C1+C2]."""
    _c(prev, torch.bfloat16, "prev")
    _c(skip, torch.bfloat16, "skip")
    n, ph, pw, C1 = prev.shape
    n2, H, W, C2 = skip.shape
    if n != n2 or tuple(out.shape) != (n, H, W, C1 + C2):
        raise LavtError("upsample_concat: shape mismatch")
    check(lib().lavt_upsample_concat(prev.data_ptr(), ph, pw, C1, skip.data_ptr(), C2,
                                     _c(out, torch.bfloat16, "out").data_ptr(), n, H, W, stream_ptr()),
          "lavt_upsample_concat")


def upconv_blend(z, p, s, b, out) -> None:
    """z bf16 [n,h,w,9*hid] (Z = Y . W_tap on the coarse map); p fp32 [n,H,W,hid] or None; s, b fp32 [hid]; out bf16 [n,H,W,hid]
    = ReLU((p if given, else b) + s * conv3x3 of the bilinear (align_corners) upsample, assembled from z)."""
    n, h, w, c9 = _c(z, torch.bfloat16, "z").shape
    n2, H, W, hid = _c(out, torch.bfloat16, "out").shape
    if n != n2 or c9 != 9 * hid or tuple(s.shape) != (hid,) or tuple(b.shape) != (hid,) or (p is not None and tuple(p.shape) != (n, H, W, hid)):
        raise LavtError("upconv_blend: shape mismatch")
    t0 = TIMER.begin()
    check(lib().lavt_upconv_blend(z.data_ptr(), h, w, hid, None if p is None else _c(p, torch.float32, "p").data_ptr(),
                                  _c(s, torch.float32, "s").data_ptr(), _c(b, torch.float32, "b").data_ptr(), out.data_ptr(),
                                  n, H, W, stream_ptr()), "lavt_upconv_blend")
    TIMER.end(t0, "upconv_blend_kernel", 2.0 * 36 * n * H * W * hid, 2.0 * z.numel() + 2.0 * out.numel() + (4.0 * p.numel() if p is not None else 0.0),
              f"{n}x{h}x{w} -> {H}x{W} hid{hid}")


def conv1x1_logits(y, w, b, out) -> None:
    """y bf16 [npix, C]; w fp32 [2, C]; b fp32 [2]; out fp32 [npix, 2]."""
    _c(y, torch.bfloat16, "y")
    npix, Cn = y.shape
    check(lib().lavt_conv1x1_logits(y.data_ptr(), _c(w, torch.float32, "w").data_ptr(), _c(b, torch.float32, "b").data_ptr(),
                                    _c(out, torch.float32, "out").data_ptr(), npix, Cn, stream_ptr()), "lavt_conv1x1_logits")


def upsample_logits(inp, out) -> None:
    """inp fp32 [n,h,w,2] -> out fp32 [n,2,H,W]."""
    n, h, w, two = inp.shape
    n2, two2, H, W = out.shape
    if two != 2 or two2 != 2 or n != n2:
        raise LavtError("upsample_logits: shape mismatch")
    check(lib().lavt_upsample_logits(_c(inp, torch.float32, "in").data_ptr(), _c(out, torch.float32, "out").data_ptr(),
                                     n, h, w, H, W, stream_ptr()), "lavt_upsample_logits")


def nhwc_to_nchw(inp, out) -> None:
    """inp fp32 [n,P,C] -> out fp32 [n,C,P]."""
    n, P, Cn = inp.shape
    check(lib().lavt_nhwc_to_nchw(_c(inp, torch.float32, "in").data_ptr(), _c(out, torch.float32, "out").data_ptr(),
                                  n, P, Cn, stream_ptr()), "lavt_nhwc_to_nchw")


def nchw_to_nhwc_bf16(inp, out) -> None:
    """inp fp32 [n,C,P] -> out bf16 [n,P,C]."""
    n, Cn, P = inp.shape
    check(lib().lavt_nchw_to_nhwc_bf16(_c(inp, torch.float32, "in").data_ptr(), _c(out, torch.bfloat16, "out").data_ptr(),
                                       n, P, Cn, stream_ptr()), "lavt_nchw_to_nhwc_bf16")


# ------------------------------------------------------------------------------------------------
# backward pass
# ------------------------------------------------------------------------------------------------
def splitk_workspace_floats(M: int, N: int, K: int) -> int:
    return int(lib().lavt_gemm_splitk_workspace_floats(M, N, K))


def gemm_bf16_splitk(a_t: torch.Tensor, b_t: torch.Tensor, dst: torch.Tensor, workspace: torch.Tensor, *, accumulate: bool = True,
                     b_koff: int = 0, K: Optional[int] = None) -> None:
    """dst[M, N] (+)= a_t[M, K] @ b_t[N, K].T with split-K; a_t / b_t bf16 (K-major), dst fp32 (row pitch dst.stride(0))."""
    _req(a_t, torch.bfloat16, "a_t")
    _req(b_t, torch.bfloat16, "b_t")
    _req(dst, torch.float32, "dst")
    M = a_t.shape[0]
    N = b_t.shape[0]
    K = int(K if K is not None else a_t.shape[1])
    if tuple(dst.shape) != (M, N):
        raise LavtError(f"split-K gemm: dst shape {tuple(dst.shape)} != ({M}, {N})")
    t0 = TIMER.begin()
    check(lib().lavt_gemm_bf16_splitk(a_t.data_ptr(), a_t.stride(0), b_t.data_ptr(), b_t.stride(0), M, N, K, b_koff,
                                      _c(workspace, torch.float32, "workspace").data_ptr(), workspace.numel(), dst.data_ptr(),
                                      dst.stride(0), 1 if accumulate else 0, stream_ptr()), "lavt_gemm_bf16_splitk")
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * M * N * K, 2.0 * (M * K + N * K) + 4.0 * M * N, f"wgrad M{M} N{N} K{K}")


def gemm_bf16_wgrad(dy: torch.Tensor, x: torch.Tensor, dst: torch.Tensor, workspace: torch.Tensor, *, accumulate: bool = True) -> None:
    """dst[out, in] (+)= dy[tokens, out].T @ x[tokens, in] from the row-major activations (MN-major tcgen05 operands, split-K)."""
    _req(dy, torch.bfloat16, "dy")
    _req(x, torch.bfloat16, "x")
    _req(dst, torch.float32, "dst")
    tokens, n_out = dy.shape
    n_in = x.shape[1]
    if x.shape[0] != tokens or tuple(dst.shape) != (n_out, n_in):
        raise LavtError("wgrad gemm: shape mismatch")
    t0 = TIMER.begin()
    check(lib().lavt_gemm_bf16_wgrad(dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0), tokens, n_out, n_in,
                                     _c(workspace, torch.float32, "workspace").data_ptr(), workspace.numel(), dst.data_ptr(),
                                     dst.stride(0), 1 if accumulate else 0, stream_ptr()), "lavt_gemm_bf16_wgrad")
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * tokens * n_out * n_in, 2.0 * tokens * (n_out + n_in) + 4.0 * n_out * n_in,
              f"wgrad-mn tokens{tokens} out{n_out} in{n_in}")


def conv3x3_wgrad_workspace_floats(n_img: int, H: int, W: int, Cin: int, Cout: int) -> int:
    return int(lib().lavt_conv3x3_wgrad_workspace_floats(n_img, H, W, Cin, Cout))


def conv3x3_wgrad(dz_nhwc: torch.Tensor, x_nhwc: torch.Tensor, dw_taps: torch.Tensor, workspace: torch.Tensor, *, accumulate: bool = True) -> None:
    """dw_taps fp32 [Cout, 9*Cin] (+)= conv3x3 weight gradient from dz bf16 [n,H,W,Cout] and x bf16 [n,H,W,Cin] (both contiguous NHWC)."""
    _c(dz_nhwc, torch.bfloat16, "dz")
    _c(x_nhwc, torch.bfloat16, "x")
    n, H, W, Cout = dz_nhwc.shape
    Cin = x_nhwc.shape[-1]
    if tuple(x_nhwc.shape[:3]) != (n, H, W) or tuple(dw_taps.shape) != (Cout, 9 * Cin):
        raise LavtError("conv3x3_wgrad: shape mismatch")
    t0 = TIMER.begin()
    check(lib().lavt_conv3x3_wgrad(dz_nhwc.data_ptr(), x_nhwc.data_ptr(), n, H, W, Cin, Cout, _c(workspace, torch.float32, "workspace").data_ptr(),
                                   workspace.numel(), _c(dw_taps, torch.float32, "dw_taps").data_ptr(), 1 if accumulate else 0, stream_ptr()),
          "lavt_conv3x3_wgrad")
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * n * H * W * Cout * 9 * Cin, 2.0 * n * H * W * (Cout + Cin) + 4.0 * Cout * 9 * Cin,
              f"conv-wgrad {n}x{H}x{W} Cin{Cin} Cout{Cout}")


def conv3d_wgrad(dz_ndhwc: torch.Tensor, x_ndhwc: torch.Tensor, dw_taps: torch.Tensor, ws_get, *, accumulate: bool = True) -> None:
    """dw_taps fp32 [Cout, 27*Cin] (+)= Conv3d(3,3,3) weight gradient from dz bf16 [B,D,H,W,Cout] and x bf16 [B,D,H,W,Cin] (contiguous);
    ``ws_get(n_floats)`` returns an fp32 workspace tensor of at least that many elements."""
    _c(dz_ndhwc, torch.bfloat16, "dz")
    _c(x_ndhwc, torch.bfloat16, "x")
    B, D, H, W, Cout = dz_ndhwc.shape
    Cin = x_ndhwc.shape[-1]
    if tuple(x_ndhwc.shape[:4]) != (B, D, H, W) or tuple(dw_taps.shape) != (Cout, 27 * Cin):
        raise LavtError("conv3d_wgrad: shape mismatch")
    workspace = ws_get(int(lib().lavt_conv3d_wgrad_workspace_floats(B, D, H, W, Cin, Cout)))
    t0 = TIMER.begin()
    check(lib().lavt_conv3d_wgrad(dz_ndhwc.data_ptr(), x_ndhwc.data_ptr(), B, D, H, W, Cin, Cout, _c(workspace, torch.float32, "workspace").data_ptr(),
                                  workspace.numel(), _c(dw_taps, torch.float32, "dw_taps").data_ptr(), 1 if accumulate else 0, stream_ptr()),
          "lavt_conv3d_wgrad")
    TIMER.end(t0, "gemm_bf16_tc_kernel", 2.0 * B * D * H * W * Cout * 27 * Cin, 2.0 * B * D * H * W * (Cout + Cin) + 4.0 * Cout * 27 * Cin,
              f"conv3d-wgrad {B}x{D}x{H}x{W} Cin{Cin} Cout{Cout}")


def transpose_bf16(x: torch.Tensor, out: torch.Tensor) -> None:
    """x bf16 [M, N] -> out bf16 [N, M] (row pitches taken from the tensors)."""
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    M, N = x.shape
    if tuple(out.shape) != (N, M):
        raise LavtError("transpose: shape mismatch")
    check(lib().lavt_transpose_bf16(x.data_ptr(), x.stride(0), out.data_ptr(), out.stride(0), M, N, stream_ptr()), "lavt_transpose_bf16")


def colsum_accumulate(x: torch.Tensor, dst: torch.Tensor) -> None:
    """dst[n] += sum_m x[m, n]; x bf16 or fp32 [M, N]."""
    if x.dtype not in (torch.bfloat16, torch.float32):
        raise LavtError("colsum: x must be bf16 or fp32")
    _req(x, x.dtype, "x")
    M, N = x.shape
    check(lib().lavt_colsum_accumulate(x.data_ptr(), 1 if x.dtype == torch.bfloat16 else 0, x.stride(0), M, N,
                                       _c(dst, torch.float32, "dst").data_ptr(), stream_ptr()), "lavt_colsum_accumulate")


def cast_rows_bf16(x: torch.Tensor, out: torch.Tensor, geom: Optional[WinGeom] = None, rscale: Optional[torch.Tensor] = None,
                   rscale_rows: int = 0, colsum: Optional[torch.Tensor] = None) -> None:
    """out bf16 [M, C] = x fp32 rows (identity) or gathered into window order (pad rows zero), optionally times a per-sample scale
    rscale[source row // rscale_rows] (DropPath backward).  ``colsum`` fp32 [C]: the column sums of the written values are added
    into it by the same pass (the bias gradient of the layer whose output gradient this is)."""
    _req(x, torch.float32, "x")
    M, Cn = out.shape
    if colsum is not None:
        check(lib().lavt_cast_rows_colsum_bf16(x.data_ptr(), x.stride(0), M, Cn, C.byref(geom) if geom is not None else None,
                                               ptr(rscale), int(rscale_rows), _c(out, torch.bfloat16, "out").data_ptr(),
                                               _c(colsum, torch.float32, "colsum").data_ptr(), stream_ptr()), "lavt_cast_rows_colsum_bf16")
        return
    check(lib().lavt_cast_rows_scaled_bf16(x.data_ptr(), x.stride(0), M, Cn, C.byref(geom) if geom is not None else None,
                                           ptr(rscale), int(rscale_rows), _c(out, torch.bfloat16, "out").data_ptr(), stream_ptr()),
          "lavt_cast_rows_scaled_bf16")


def gelu_fwd(x: torch.Tensor, y: torch.Tensor) -> None:
    check(lib().lavt_gelu_fwd(_c(x, torch.bfloat16, "x").data_ptr(), _c(y, torch.bfloat16, "y").data_ptr(), x.numel(), stream_ptr()),
          "lavt_gelu_fwd")


def gelu_bwd(dy: torch.Tensor, x: torch.Tensor, dx: torch.Tensor) -> None:
    check(lib().lavt_gelu_bwd(_c(dy, torch.bfloat16, "dy").data_ptr(), _c(x, torch.bfloat16, "x").data_ptr(),
                              _c(dx, torch.bfloat16, "dx").data_ptr(), x.numel(), stream_ptr()), "lavt_gelu_bwd")


def layernorm_rows_bwd(x, dy, gamma, dx, dgamma, dbeta, *, dres=None, eps: float = 1e-5) -> None:
    """x fp32 [M, C] (LN input), dy bf16 [M, C]; dx fp32 [M, C] = (dres or 0) + LN'(dy); dgamma / dbeta fp32 [C] accumulate."""
    _req(x, torch.float32, "x")
    M, Cn = x.shape
    _req(dy, torch.bfloat16, "dy")
    check(lib().lavt_layernorm_rows_bwd(x.data_ptr(), x.stride(0), M, Cn, dy.data_ptr(), dy.stride(0),
                                        _c(gamma, torch.float32, "gamma").data_ptr(), eps, ptr(dres), _c(dx, torch.float32, "dx").data_ptr(),
                                        _c(dgamma, torch.float32, "dgamma").data_ptr(), _c(dbeta, torch.float32, "dbeta").data_ptr(),
                                        stream_ptr()), "lavt_layernorm_rows_bwd")


def layernorm_window_gather_bwd(x, geom: WinGeom, dy, gamma, dx, dgamma, dbeta, *, dres=None, eps: float = 1e-5) -> None:
    """x fp32 [tokens, C]; dy bf16 [geom.rows(), C] in window order."""
    _c(x, torch.float32, "x")
    Cn = x.shape[-1]
    check(lib().lavt_layernorm_window_gather_bwd(x.data_ptr(), Cn, C.byref(geom), _c(dy, torch.bfloat16, "dy").data_ptr(),
                                                 _c(gamma, torch.float32, "gamma").data_ptr(), eps, ptr(dres),
                                                 _c(dx, torch.float32, "dx").data_ptr(), _c(dgamma, torch.float32, "dgamma").data_ptr(),
                                                 _c(dbeta, torch.float32, "dbeta").data_ptr(), stream_ptr()),
          "lavt_layernorm_window_gather_bwd")


def patch_merge_layernorm_bwd(x, B, D, H, W, dy, gamma, dx, dgamma, dbeta, eps: float = 1e-5) -> None:
    """x fp32 [B*D*H*W, C]; dy bf16 [B*D*ceil(H/2)*ceil(W/2), 4C]; dx fp32 like x (every token written exactly once)."""
    _c(x, torch.float32, "x")
    Cn = x.shape[-1]
    check(lib().lavt_patch_merge_layernorm_bwd(x.data_ptr(), B, D, H, W, Cn, _c(dy, torch.bfloat16, "dy").data_ptr(),
                                               _c(gamma, torch.float32, "gamma").data_ptr(), eps, _c(dx, torch.float32, "dx").data_ptr(),
                                               _c(dgamma, torch.float32, "dgamma").data_ptr(), _c(dbeta, torch.float32, "dbeta").data_ptr(),
                                               stream_ptr()), "lavt_patch_merge_layernorm_bwd")


def window_attention_bwd(qkv, out, dout, table_t, geom: WinGeom, dqkv, dtable_t, lse=None, workspace=None) -> None:
    """Adjoint of window_attention; dtable_t fp32 [nH, L] accumulates (or None); lse = the forward's row statistics or None
    (recomputed).  workspace: fp32 scratch of at least window_attention_bwd_workspace_floats(table_t, geom) elements, or None: then
    one is allocated here when this geometry needs it (pass a reused buffer for CUDA-graph capture)."""
    nH, L = table_t.shape
    if workspace is None:
        need = window_attention_bwd_workspace_floats(table_t, geom) if lse is not None else 0
        if need > 0:
            workspace = torch.empty(need, dtype=torch.float32, device=qkv.device)
    t0 = TIMER.begin()
    check(lib().lavt_window_attention_bwd(_c(qkv, torch.bfloat16, "qkv").data_ptr(), _c(out, torch.bfloat16, "out").data_ptr(),
                                          _c(dout, torch.bfloat16, "dout").data_ptr(), _c(table_t, torch.float32, "table_t").data_ptr(),
                                          L, nH, C.byref(geom), ptr(lse), _c(dqkv, torch.bfloat16, "dqkv").data_ptr(),
                                          ptr(dtable_t), None if workspace is None else _c(workspace, torch.float32, "workspace").data_ptr(),
                                          0 if workspace is None else workspace.numel(), stream_ptr()),
          "lavt_window_attention_bwd")
    rows = geom.rows()
    TIMER.end(t0, "window_attn_bwd_kernel", 12.0 * rows * geom.N * nH * 32, 2.0 * rows * nH * 32 * 8, f"rows{rows} N{geom.N} nH{nH}")


def pwam_attend_bwd(qpre, stats, k, v, mask, do, dqhat, qs, p_bd, ds_bd, sums, heads: int, nl_pad: int) -> None:
    B, n, Cn = qpre.shape
    Nl = k.shape[1]
    if tuple(p_bd.shape) != (B * n, B * heads * nl_pad) or tuple(ds_bd.shape) != tuple(p_bd.shape):
        raise LavtError("pwam_attend_bwd: block-diagonal buffers have the wrong shape")
    check(lib().lavt_pwam_attend_bwd(_c(qpre, torch.float32, "qpre").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                     _c(k, torch.float32, "k").data_ptr(), _c(v, torch.float32, "v").data_ptr(),
                                     _c(mask, torch.float32, "mask").data_ptr(), _c(do, torch.bfloat16, "do").data_ptr(),
                                     _c(dqhat, torch.float32, "dqhat").data_ptr(), _c(qs, torch.bfloat16, "qs").data_ptr(),
                                     _c(p_bd, torch.bfloat16, "p_bd").data_ptr(), _c(ds_bd, torch.bfloat16, "ds_bd").data_ptr(),
                                     _c(sums, torch.float32, "sums").data_ptr(), B, n, Cn, Nl, nl_pad, heads, stream_ptr()),
          "lavt_pwam_attend_bwd")


def pwam_mul_norm_bwd(da2, vis, vispre, langpre, stats, dvispre, sums) -> None:
    B, n, Cn = langpre.shape
    check(lib().lavt_pwam_mul_norm_bwd(_c(da2, torch.bfloat16, "da2").data_ptr(), _c(vis, torch.bfloat16, "vis").data_ptr(),
                                       _c(vispre, torch.bfloat16, "vispre").data_ptr(), _c(langpre, torch.float32, "langpre").data_ptr(),
                                       _c(stats, torch.float32, "stats").data_ptr(), _c(dvispre, torch.bfloat16, "dvispre").data_ptr(),
                                       _c(sums, torch.float32, "sums").data_ptr(), B, n, Cn, stream_ptr()), "lavt_pwam_mul_norm_bwd")


def instnorm_bwd(xpre, stats, sums, out, *, g_f32=None, ga=None, gb=None) -> None:
    B, n, Cn = xpre.shape
    check(lib().lavt_instnorm_bwd(ptr(g_f32), ptr(ga), ptr(gb), _c(xpre, torch.float32, "xpre").data_ptr(),
                                  _c(stats, torch.float32, "stats").data_ptr(), _c(sums, torch.float32, "sums").data_ptr(),
                                  _c(out, torch.bfloat16, "out").data_ptr(), B, n, Cn, stream_ptr()), "lavt_instnorm_bwd")


def pwam_kv_bwd(dkbuf, dvbuf, mask, l, wk, wv, dwk, dbk, dwv, dbv, dl, heads: int, nl_pad: int) -> None:
    B, Lin, Nl = l.shape
    Cn = wk.shape[0]
    check(lib().lavt_pwam_kv_bwd(_c(dkbuf, torch.float32, "dkbuf").data_ptr(), _c(dvbuf, torch.float32, "dvbuf").data_ptr(),
                                 _c(mask, torch.float32, "mask").data_ptr(), _c(l, torch.float32, "l").data_ptr(),
                                 _c(wk, torch.float32, "wk").data_ptr(), _c(wv, torch.float32, "wv").data_ptr(), ptr(dwk), ptr(dbk),
                                 ptr(dwv), ptr(dbv), ptr(dl), B, Nl, nl_pad, Lin, Cn, heads, stream_ptr()), "lavt_pwam_kv_bwd")


def gate_elementwise(mode: int, a, b=None, f=None, f2=None, out_bf16=None, out_f32=None) -> None:
    check(lib().lavt_gate_elementwise(mode, _c(a, torch.bfloat16, "a").data_ptr(), ptr(b), ptr(f), ptr(f2), ptr(out_bf16), ptr(out_f32),
                                      a.numel(), stream_ptr()), "lavt_gate_elementwise")


# ---- SimpleDecoding (training mode), final upsample and loss ----
def bn_relu_apply(z, stats, gamma, beta, t) -> None:
    """z fp32 [npix, C]; stats fp32 [2, C] (mean, rstd); t bf16 [npix, C]."""
    npix, Cn = z.shape
    check(lib().lavt_bn_relu_apply(_c(z, torch.float32, "z").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                   _c(gamma, torch.float32, "gamma").data_ptr(), _c(beta, torch.float32, "beta").data_ptr(),
                                   _c(t, torch.bfloat16, "t").data_ptr(), npix, Cn, stream_ptr()), "lavt_bn_relu_apply")


def bn_relu_bwd_reduce(dt, t, z, stats, sums) -> None:
    npix, Cn = z.shape
    check(lib().lavt_bn_relu_bwd_reduce(_c(dt, torch.bfloat16, "dt").data_ptr(), _c(t, torch.bfloat16, "t").data_ptr(),
                                        _c(z, torch.float32, "z").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                        _c(sums, torch.float32, "sums").data_ptr(), npix, Cn, stream_ptr()), "lavt_bn_relu_bwd_reduce")


def bn_relu_bwd_apply(dt, t, z, stats, gamma, sums, dz, n_stat: int) -> None:
    npix, Cn = z.shape
    check(lib().lavt_bn_relu_bwd_apply(_c(dt, torch.bfloat16, "dt").data_ptr(), _c(t, torch.bfloat16, "t").data_ptr(),
                                       _c(z, torch.float32, "z").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                       _c(gamma, torch.float32, "gamma").data_ptr(), _c(sums, torch.float32, "sums").data_ptr(),
                                       _c(dz, torch.bfloat16, "dz").data_ptr(), npix, n_stat, Cn, stream_ptr()), "lavt_bn_relu_bwd_apply")


def instnorm_bwd_reduce(g, xpre, stats, sums) -> None:
    """sums fp32 [B,2,C] += (sum_n g, sum_n g * IN(xpre)); g, xpre fp32 [B,n,C]."""
    B, n, Cn = xpre.shape
    check(lib().lavt_instnorm_bwd_reduce(_c(g, torch.float32, "g").data_ptr(), _c(xpre, torch.float32, "xpre").data_ptr(),
                                         _c(stats, torch.float32, "stats").data_ptr(), _c(sums, torch.float32, "sums").data_ptr(),
                                         B, n, Cn, stream_ptr()), "lavt_instnorm_bwd_reduce")


def nhwc_pad_transpose(x_nhwc, out, wp: int, dshift: int = 0, frames_per_clip: int = 0) -> None:
    """x bf16 [n,H,W,C] (last dim contiguous, pixel pitch x.stride(2)) -> out bf16 [C, >= n*(H+2)*wp], pre-zeroed by the caller;
    pixel (img,h,w) lands in column (img*(H+2) + h+1)*wp + w+1 - dshift; with frames_per_clip = D > 0 the images are frames of clips that
    get a zero frame on either side (img -> clip*(D+2) + d+1)."""
    _req(x_nhwc, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    n, H, W, Cn = x_nhwc.shape
    check(lib().lavt_nhwc_pad_transpose(x_nhwc.data_ptr(), x_nhwc.stride(2), out.data_ptr(), out.stride(0),
                                        n, H, W, Cn, wp, dshift, frames_per_clip, stream_ptr()), "lavt_nhwc_pad_transpose")


def upsample_concat_bwd(dcat, dprev) -> None:
    """dcat bf16 [n,H,W,Ct] -> dprev bf16 [n,ph,pw,C1] (gradient of the upsampled first C1 channels)."""
    n, H, W, Ct = dcat.shape
    n2, ph, pw, C1 = dprev.shape
    check(lib().lavt_upsample_concat_bwd(_c(dcat, torch.bfloat16, "dcat").data_ptr(), Ct, _c(dprev, torch.bfloat16, "dprev").data_ptr(),
                                         ph, pw, C1, n, H, W, stream_ptr()), "lavt_upsample_concat_bwd")


def conv1x1_logits_bwd(dlogits, y, w, dy, dw, db) -> None:
    npix, Cn = y.shape
    check(lib().lavt_conv1x1_logits_bwd(_c(dlogits, torch.float32, "dlogits").data_ptr(), _c(y, torch.bfloat16, "y").data_ptr(),
                                        _c(w, torch.float32, "w").data_ptr(), _c(dy, torch.bfloat16, "dy").data_ptr(),
                                        _c(dw, torch.float32, "dw").data_ptr(), _c(db, torch.float32, "db").data_ptr(), npix, Cn,
                                        stream_ptr()), "lavt_conv1x1_logits_bwd")


def upsample_logits_bwd(dout, din) -> None:
    """dout fp32 [n,2,H,W] -> din fp32 [n,h,w,2]."""
    n, _, H, W = dout.shape
    n2, h, w, _ = din.shape
    check(lib().lavt_upsample_logits_bwd(_c(dout, torch.float32, "dout").data_ptr(), _c(din, torch.float32, "din").data_ptr(), n, h, w, H, W,
                                         stream_ptr()), "lavt_upsample_logits_bwd")


def cross_entropy(logits, target, acc, dlogits=None, *, w0: float = 0.9, w1: float = 1.1, gscale: float = 1.0, phase: int = 0) -> None:
    """logits fp32 [n,2,H,W]; target int64 [n,H,W]; acc fp32 [2] (sum w*nll, sum w)."""
    n, two, H, W = logits.shape
    if target.dtype != torch.int64 or not target.is_cuda or not target.is_contiguous():
        raise LavtError("cross_entropy: target must be a contiguous CUDA int64 tensor")
    check(lib().lavt_cross_entropy(_c(logits, torch.float32, "logits").data_ptr(), target.data_ptr(), w0, w1,
                                   _c(acc, torch.float32, "acc").data_ptr(), ptr(dlogits), gscale, n, H, W, phase, stream_ptr()),
          "lavt_cross_entropy")


# ---- input / output edges ----
IMAGENET_MEAN, IMAGENET_STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def normalize_u8(frames: torch.Tensor, out: Optional[torch.Tensor] = None, mean=IMAGENET_MEAN, std=IMAGENET_STD) -> torch.Tensor:
    """T.ToTensor() + T.Normalize (reference train.py:54-60): uint8 CUDA frames [n,H,W,3] -> fp32 [n,3,H,W]."""
    if frames.dtype != torch.uint8 or not frames.is_cuda or not frames.is_contiguous() or frames.shape[-1] != 3:
        raise LavtError("normalize_u8: frames must be a contiguous CUDA uint8 tensor [n,H,W,3]")
    n, H, W, _ = frames.shape
    if out is None:
        out = torch.empty(n, 3, H, W, device=frames.device, dtype=torch.float32)
    m, s_ = (C.c_float * 3)(*mean), (C.c_float * 3)(*std)
    check(lib().lavt_normalize_u8(frames.data_ptr(), _c(out, torch.float32, "out").data_ptr(), n, H, W, C.cast(m, C.c_void_p),
                                  C.cast(s_, C.c_void_p), stream_ptr()), "lavt_normalize_u8")
    return out


def logits_to_mask(logits: torch.Tensor, size) -> torch.Tensor:
    """F.interpolate(logits, size, 'bilinear', align_corners=True).argmax(1) as the 0 / 255 uint8 image the reference saves
    (test_ytvos.py:249-253, 274-279): logits fp32 [n,2,H,W] -> uint8 [n,oh,ow]."""
    n, two, H, W = logits.shape
    if two != 2:
        raise LavtError("logits_to_mask: expects 2 classes")
    oh, ow = int(size[0]), int(size[1])
    out = torch.empty(n, oh, ow, device=logits.device, dtype=torch.uint8)
    check(lib().lavt_logits_to_mask(_c(logits, torch.float32, "logits").data_ptr(), out.data_ptr(), n, H, W, oh, ow, stream_ptr()),
          "lavt_logits_to_mask")
    return out


def gacd_fuse(xm, lang_stats, wq, bq, wc, bc, wd, bd, wv, bv, ws_get, out_f32=None, out_bf16=None) -> None:
    """GA-CD after mm_gen: xm fp32 [B,n,C]; weights fp32; ``ws_get(n_floats)`` returns an fp32 workspace."""
    B, n, Cn = xm.shape
    work = ws_get(int(lib().lavt_gacd_workspace_floats(B, n, Cn)))
    for t, nm in ((xm, "xm"), (lang_stats, "lang_stats"), (wq, "wq"), (bq, "bq"), (wc, "wc"), (bc, "bc"), (wd, "wd"), (bd, "bd"), (wv, "wv"), (bv, "bv")):
        _c(t, torch.float32, nm)
    check(lib().lavt_gacd_fuse(xm.data_ptr(), lang_stats.data_ptr(), wq.data_ptr(), bq.data_ptr(), wc.data_ptr(), bc.data_ptr(), wd.data_ptr(),
                               bd.data_ptr(), wv.data_ptr(), bv.data_ptr(), _c(work, torch.float32, "workspace").data_ptr(), ptr(out_f32),
                               ptr(out_bf16), B, n, Cn, stream_ptr()), "lavt_gacd_fuse")


def bcam_words(l: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, lr: torch.Tensor, lrT: torch.Tensor, mask: Optional[torch.Tensor] = None,
               act: int = ACT_NONE) -> None:
    """lr = lang_reduce(l^T) (reference lib/bcam.py:47): l fp32 [B,Lin,Nl], w fp32 [C,Lin] -> lr bf16 [B,Nlp,C] (pad rows zero), lrT bf16 [B,C,Nlp].
    With ``act=ACT_GELU`` and ``mask`` fp32 [B,Nl]: EFN's lang = gelu(lang_project(l)) * l_mask (:186-187)."""
    B, Lin, Nl = l.shape
    _, Nlp, Cn = lr.shape
    if tuple(lrT.shape) != (B, Cn, Nlp) or tuple(w.shape) != (Cn, Lin):
        raise LavtError("bcam_words: shape mismatch")
    check(lib().lavt_bcam_words(_c(l, torch.float32, "l").data_ptr(), _c(w, torch.float32, "w").data_ptr(), _c(bias, torch.float32, "bias").data_ptr(),
                                _c(mask, torch.float32, "mask").data_ptr() if mask is not None else None, int(act),
                                _c(lr, torch.bfloat16, "lr").data_ptr(), _c(lrT, torch.bfloat16, "lrT").data_ptr(), B, Nl, Nlp, Lin, Cn, stream_ptr()),
          "lavt_bcam_words")


def bcam_softmax_rows(s: torch.Tensor, cols: int, p: torch.Tensor, mask: Optional[torch.Tensor] = None, rows_per_mask: int = 0) -> None:
    """p[r, :cols] = softmax(s[r, :cols] + (1e4 mask - 1e4)) in bf16, p[r, cols:] = 0; s fp32 [rows, lds], p bf16 [rows, ldp], mask fp32 [*, cols]."""
    _req(s, torch.float32, "s")
    _req(p, torch.bfloat16, "p")
    rows = s.shape[0]
    if p.shape[0] != rows or s.stride(1) != 1 or p.stride(1) != 1 or s.shape[1] < cols or p.shape[1] < cols:
        raise LavtError("bcam_softmax_rows: shape mismatch")
    if mask is not None:
        _c(mask, torch.float32, "mask")
        if mask.shape[-1] != cols or rows_per_mask <= 0 or mask.numel() // cols * rows_per_mask < rows:
            raise LavtError("bcam_softmax_rows: mask shape mismatch")
    check(lib().lavt_bcam_softmax_rows(s.data_ptr(), s.stride(0), ptr(mask), int(rows_per_mask), p.data_ptr(), p.stride(0), rows, int(cols),
                                       stream_ptr()), "lavt_bcam_softmax_rows")


def bcam_transpose_pad(x: torch.Tensor, out: torch.Tensor) -> None:
    """x bf16 [B*n, C] (row pitch x.stride(0)) -> out bf16 [B, C, ldo >= n], columns n.. zero."""
    _req(x, torch.bfloat16, "x")
    B, Cn, ldo = out.shape
    n = x.shape[0] // B
    if x.shape[0] != B * n or x.shape[1] != Cn or x.stride(1) != 1 or ldo < n:
        raise LavtError("bcam_transpose_pad: shape mismatch")
    check(lib().lavt_bcam_transpose_pad(x.data_ptr(), x.stride(0), _c(out, torch.bfloat16, "out").data_ptr(), ldo, B, n, Cn, stream_ptr()),
          "lavt_bcam_transpose_pad")


def efn_sentence_bias(l: torch.Tensor, mask: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, sb: torch.Tensor) -> None:
    """sb fp32 [B,C] = bias + w @ masked-mean(l) (reference lib/bcam.py:179-185); l fp32 [B,Lin,Nl], mask fp32 [B,Nl], w fp32 [C,Lin] (row pitch free)."""
    B, Lin, Nl = l.shape
    _req(w, torch.float32, "w")
    Cn = w.shape[0]
    if w.shape[1] != Lin or tuple(sb.shape) != (B, Cn) or tuple(mask.shape) != (B, Nl):
        raise LavtError("efn_sentence_bias: shape mismatch")
    check(lib().lavt_efn_sentence_bias(_c(l, torch.float32, "l").data_ptr(), _c(mask, torch.float32, "mask").data_ptr(), w.data_ptr(), w.stride(0),
                                       _c(bias, torch.float32, "bias").data_ptr(), _c(sb, torch.float32, "sb").data_ptr(), B, Nl, Lin, Cn,
                                       stream_ptr()), "lavt_efn_sentence_bias")


def efn_norm_pool(pre: torch.Tensor, stats: torch.Tensor, out: torch.Tensor, h: int, pool: bool) -> None:
    """out bf16 [B, rows_out, C] = (2 x 2 average pool of) InstanceNorm(pre fp32 [B,n,C]) with stats fp32 [B,2,C]; surplus rows zero."""
    B, n, Cn = pre.shape
    if out.shape[0] != B or out.shape[2] != Cn:
        raise LavtError("efn_norm_pool: shape mismatch")
    check(lib().lavt_efn_norm_pool(_c(pre, torch.float32, "pre").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(),
                                   _c(out, torch.bfloat16, "out").data_ptr(), B, n, int(h), 1 if pool else 0, out.shape[1], Cn, stream_ptr()),
          "lavt_efn_norm_pool")


def efn_norm_upsample(pre: torch.Tensor, stats: torch.Tensor, n: int, h: int, up: bool, out_f32=None, out_bf16=None) -> None:
    """out [B*n, C] = (bilinear x 2, align_corners False, of) InstanceNorm(pre fp32 [B, n/4 or n, C])."""
    B, n_in, Cn = pre.shape
    if n_in != (n // 4 if up else n):
        raise LavtError("efn_norm_upsample: shape mismatch")
    for t, dt, nm in ((out_f32, torch.float32, "out_f32"), (out_bf16, torch.bfloat16, "out_bf16")):
        if t is not None:
            _c(t, dt, nm)
            if t.numel() != B * n * Cn:
                raise LavtError("efn_norm_upsample: output size mismatch")
    check(lib().lavt_efn_norm_upsample(_c(pre, torch.float32, "pre").data_ptr(), _c(stats, torch.float32, "stats").data_ptr(), ptr(out_f32),
                                       ptr(out_bf16), B, n, int(h), 1 if up else 0, Cn, stream_ptr()), "lavt_efn_norm_upsample")


def efn_word_attend(score: torch.Tensor, mask: torch.Tensor, g: torch.Tensor, out: torch.Tensor) -> None:
    """out fp32 [B*n, C] = softmax(score[:, :Nl] + (1e4 mask - 1e4)) @ g[b]; score fp32 [B*n, lds], mask fp32 [B,Nl], g fp32 [B, g_rows >= Nl, C]."""
    _req(score, torch.float32, "score")
    B, Nl = mask.shape
    rows = score.shape[0]
    Cn = g.shape[2]
    if rows % B or g.shape[0] != B or g.shape[1] < Nl or score.shape[1] < Nl or tuple(out.shape) != (rows, Cn):
        raise LavtError("efn_word_attend: shape mismatch")
    check(lib().lavt_efn_word_attend(score.data_ptr(), score.stride(0), _c(mask, torch.float32, "mask").data_ptr(), _c(g, torch.float32, "g").data_ptr(),
                                     g.shape[1], _c(out, torch.float32, "out").data_ptr(), B, rows // B, Nl, Cn, stream_ptr()), "lavt_efn_word_attend")


# ---- VLT head glue (csrc/vlt_kernels.cu) ----
def _rows2d(t: torch.Tensor, name: str) -> torch.Tensor:
    if not t.is_cuda or t.dim() != 2 or t.stride(1) != 1:
        raise LavtError(f"{name} must be a 2-D CUDA tensor with contiguous rows (no CPU fallback)")
    return t


def rows_affine_act(x: torch.Tensor, *, add: Optional[torch.Tensor] = None, v: Optional[torch.Tensor] = None, rows_per_image: int = 0,
                    s: Optional[torch.Tensor] = None,
                    t: Optional[torch.Tensor] = None, act: int = ACT_NONE, out_bf16: Optional[torch.Tensor] = None,
                    out_f32: Optional[torch.Tensor] = None) -> None:
    """out[r, c] = act((x[r, c] + add[r, c]) * v[r // rows_per_image, c] * s[c] + t[c]); x bf16 / fp32 [rows, C] (row pitch free), add bf16."""
    _rows2d(x, "x")
    if x.dtype not in (torch.bfloat16, torch.float32):
        raise LavtError("rows_affine_act: x must be bf16 or fp32")
    rows, Cn = x.shape
    out = out_bf16 if out_bf16 is not None else out_f32
    if out is None:
        raise LavtError("rows_affine_act needs an output")
    for o, dt, nm in ((out_bf16, torch.bfloat16, "out_bf16"), (out_f32, torch.float32, "out_f32")):
        if o is not None and (_rows2d(o, nm).dtype != dt or tuple(o.shape) != (rows, Cn) or o.stride(0) != out.stride(0)):
            raise LavtError(f"rows_affine_act: {nm} has the wrong dtype / shape / pitch")
    for vec, nm in ((s, "s"), (t, "t")):
        if vec is not None:
            _c(vec, torch.float32, nm)
    if add is not None:
        _req(_rows2d(add, "add"), torch.bfloat16, "add")
        if tuple(add.shape) != (rows, Cn):
            raise LavtError("rows_affine_act: addend shape mismatch")
    check(lib().lavt_rows_affine_act(x.data_ptr(), 1 if x.dtype == torch.bfloat16 else 0, x.stride(0), ptr(add), add.stride(0) if add is not None else 0,
                                     _c(v, torch.float32, "v").data_ptr() if v is not None else None, int(rows_per_image), ptr(s), ptr(t), int(act),
                                     ptr(out_bf16), ptr(out_f32), out.stride(0), rows, Cn, stream_ptr()), "lavt_rows_affine_act")


def avgpool2_nhwc(x: torch.Tensor, out: torch.Tensor) -> None:
    """x bf16 [n,H,W,C] (pixel pitch x.stride(2)) -> out bf16 [n,H/2,W/2,C] (pixel pitch out.stride(2))."""
    _req(x, torch.bfloat16, "x")
    _req(out, torch.bfloat16, "out")
    n, H, W, Cn = x.shape
    if tuple(out.shape) != (n, H // 2, W // 2, Cn):
        raise LavtError("avgpool2: shape mismatch")
    check(lib().lavt_avgpool2_nhwc(x.data_ptr(), x.stride(2), out.data_ptr(), out.stride(2), n, H, W, Cn, stream_ptr()), "lavt_avgpool2_nhwc")


def append_coords(x: torch.Tensor, out: torch.Tensor) -> None:
    """x bf16 [n,H,W,C] (pixel pitch free) -> out bf16 contiguous [n,H,W,C+8] = x | xxx yyy 00 (vlt_concat_coords)."""
    _req(x, torch.bfloat16, "x")
    n, H, W, Cn = x.shape
    if tuple(out.shape) != (n, H, W, Cn + 8):
        raise LavtError("append_coords: shape mismatch")
    check(lib().lavt_append_coords(x.data_ptr(), x.stride(2), _c(out, torch.bfloat16, "out").data_ptr(), n, H, W, Cn, stream_ptr()),
          "lavt_append_coords")


def rows_add_table(x: torch.Tensor, table: torch.Tensor, *, out_bf16: Optional[torch.Tensor] = None, out_f32: Optional[torch.Tensor] = None) -> None:
    """out[r, :] = x[r, :] + table[r % table.shape[0], :]."""
    _rows2d(x, "x")
    rows, Cn = x.shape
    out = out_bf16 if out_bf16 is not None else out_f32
    if out is None or table.shape[1] != Cn:
        raise LavtError("rows_add_table: missing output / table width mismatch")
    for o in (out_bf16, out_f32):
        if o is not None and (tuple(o.shape) != (rows, Cn) or o.stride(0) != out.stride(0)):
            raise LavtError("rows_add_table: output shape / pitch mismatch")
    check(lib().lavt_rows_add_table(x.data_ptr(), 1 if x.dtype == torch.bfloat16 else 0, x.stride(0), _c(table, torch.float32, "table").data_ptr(),
                                    table.shape[0], ptr(out_bf16), ptr(out_f32), out.stride(0), rows, Cn, stream_ptr()), "lavt_rows_add_table")


def mha_small(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, B: int, heads: int, key_mask: Optional[torch.Tensor] = None) -> None:
    """q bf16 [B*Lq, >= heads*32], k / v bf16 [B*S, >= heads*32] (column windows of packed projections are fine), out bf16 [B*Lq, heads*32];
    key_mask fp32 [B, S] with 0 = ignore the key."""
    for t_, nm in ((q, "q"), (k, "k"), (v, "v"), (out, "out")):
        _req(_rows2d(t_, nm), torch.bfloat16, nm)
    Lq, S = q.shape[0] // B, k.shape[0] // B
    if q.shape[0] != B * Lq or k.shape[0] != B * S or v.shape[0] != B * S or out.shape[0] != B * Lq:
        raise LavtError("mha_small: row counts are not multiples of the batch")
    check(lib().lavt_mha_small(q.data_ptr(), q.stride(0), k.data_ptr(), k.stride(0), v.data_ptr(), v.stride(0),
                               _c(key_mask, torch.float32, "key_mask").data_ptr() if key_mask is not None else None, out.data_ptr(), out.stride(0),
                               B, Lq, S, heads, stream_ptr()), "lavt_mha_small")


def gate_transpose(x: torch.Tensor, gate: torch.Tensor, out: torch.Tensor, B: int) -> None:
    """x fp32 [B*Q, S], gate fp32 [B*Q, >=1] (first column used) -> out bf16 [B, S, Q]."""
    _req(_rows2d(x, "x"), torch.float32, "x")
    _req(_rows2d(gate, "gate"), torch.float32, "gate")
    Q, S = x.shape[0] // B, x.shape[1]
    if tuple(out.shape) != (B, S, Q):
        raise LavtError("gate_transpose: shape mismatch")
    check(lib().lavt_gate_transpose(x.data_ptr(), x.stride(0), gate.data_ptr(), gate.stride(0), _c(out, torch.bfloat16, "out").data_ptr(), B, Q, S,
                                    stream_ptr()), "lavt_gate_transpose")


def upsample_nhwc(prev: torch.Tensor, out: torch.Tensor) -> None:
    """Bilinear (align_corners=True) resize of prev bf16 [n,ph,pw,C] to out bf16 [n,H,W,C] (lavt_upsample_concat with no skip tensor)."""
    _c(prev, torch.bfloat16, "prev")
    n, ph, pw, C1 = prev.shape
    if out.shape[0] != n or out.shape[3] != C1:
        raise LavtError("upsample_nhwc: shape mismatch")
    check(lib().lavt_upsample_concat(prev.data_ptr(), ph, pw, C1, None, 0, _c(out, torch.bfloat16, "out").data_ptr(), n, out.shape[1], out.shape[2],
                                     stream_ptr()), "lavt_upsample_concat")


# ---- fp32 validation twins (csrc/fp32_ref_kernels.cu): slow CUDA-core kernels with the production epilogue / index math ----
def gemm_f32_ref(a: torch.Tensor, w: torch.Tensor, **epi) -> None:
    """out = epilogue(a @ w.T) with fp32 operands and fp32 accumulation; a [M,K] fp32, w [N,K] fp32."""
    _req(a, torch.float32, "a")
    _req(w, torch.float32, "w")
    M, Kd = a.shape
    N, K2 = w.shape
    if Kd != K2:
        raise LavtError(f"gemm_f32_ref: K mismatch {Kd} vs {K2}")
    e = make_epilogue(**epi)
    check(lib().lavt_gemm_f32_ref(a.data_ptr(), a.stride(0), w.data_ptr(), w.stride(0), M, N, Kd, C.byref(e), stream_ptr()), "lavt_gemm_f32_ref")


def window_attention_f32_ref(qkv: torch.Tensor, table_t: torch.Tensor, geom: WinGeom, out: torch.Tensor) -> None:
    nH, L = table_t.shape
    check(lib().lavt_window_attention_f32_ref(_c(qkv, torch.float32, "qkv").data_ptr(), _c(table_t, torch.float32, "table_t").data_ptr(), L, nH,
                                              C.byref(geom), _c(out, torch.float32, "out").data_ptr(), stream_ptr()), "lavt_window_attention_f32_ref")


def layernorm_window_gather_f32(x: torch.Tensor, geom: WinGeom, gamma, beta, out_f32: torch.Tensor, eps: float = 1e-5) -> None:
    check(lib().lavt_layernorm_window_gather_f32(_c(x, torch.float32, "x").data_ptr(), x.shape[-1], C.byref(geom), _c(gamma.detach(), torch.float32, "gamma").data_ptr(),
                                                 _c(beta.detach(), torch.float32, "beta").data_ptr(), float(eps), _c(out_f32, torch.float32, "out").data_ptr(),
                                                 stream_ptr()), "lavt_layernorm_window_gather_f32")


def split3_bf16(x: torch.Tensor, out: torch.Tensor) -> None:
    """x fp32 [M,K] -> out bf16 [M,3K] = hi | lo | hi (split-precision GEMM operand)."""
    _req(_rows2d(x, "x"), torch.float32, "x")
    M, Kd = x.shape
    if tuple(out.shape) != (M, 3 * Kd):
        raise LavtError("split3: shape mismatch")
    check(lib().lavt_split3_bf16(x.data_ptr(), x.stride(0), _c(out, torch.bfloat16, "out").data_ptr(), M, Kd, stream_ptr()), "lavt_split3_bf16")


def bert_attention_f32(qkv: torch.Tensor, mask: torch.Tensor, out: torch.Tensor, heads: int) -> None:
    B, Nl = mask.shape
    H = out.shape[-1]
    check(lib().lavt_bert_attention_f32(_c(qkv, torch.float32, "qkv").data_ptr(), _c(mask, torch.float32, "mask").data_ptr(),
                                        _c(out, torch.float32, "out").data_ptr(), B, Nl, H, heads, stream_ptr()), "lavt_bert_attention_f32")
