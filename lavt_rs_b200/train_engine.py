"""Training-step engine: forward with saved activations + hand-written backward on the sm_100a kernels.

The reference trains with autograd over PyTorch ops (train.py:330-360: ``loss.backward()``).  Here every forward unit of
``engine.py`` has a ``*_fwd`` twin that keeps what its adjoint needs (bf16 GEMM operands, the fp32 LayerNorm inputs) and a
``*_bwd`` that sequences the backward kernels of ``include/lavt_b200.h``:

  * activation gradients of a Linear / Conv1d(k=1):  dX = dY W        -> ``lavt_gemm_bf16`` with the transposed bf16 weight
  * weight gradients:                                 dW += dY^T X     -> ``lavt_gemm_bf16_wgrad`` (MN-major operands, split-K)
  * bias gradients:                                   db += colsum dY  -> ``lavt_colsum_accumulate``
  * LayerNorm (+ window gather / PatchMerging gather) -> ``lavt_layernorm_*_bwd``
  * window attention                                  -> ``lavt_window_attention_bwd``

The gradient on the residual stream is fp32 [tokens, C] and is updated in place from block to block.  Parameter gradients
accumulate in fp32 buffers owned by a ``GradStore`` and are handed to ``param.grad`` by ``GradStore.finalize()``.
No PyTorch math runs on this path and there is no CPU fallback.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import os

import torch

from . import _cabi as K
from . import engine as E
from .engine import Workspace, _bf16, _f32, _count
from .geometry import window_geometry


class GradStore:
    """fp32 accumulation buffers for parameter gradients (zeroed at creation = ``optimizer.zero_grad()``, train.py:352).
    Some kernels accumulate in the layout of the engine's prepared operand rather than the parameter's; those buffers carry
    a function that maps them back to the parameter's shape when the gradients are handed over."""

    def __init__(self, params=None):
        """``params``: the parameters that will receive gradients.  Their buffers are then views of ONE zero-filled allocation
        (one memset per step instead of ~450 tiny fill kernels: the ncu launch list of a step showed 1 354 FillFunctor launches)."""
        self._g: Dict[int, Tuple[torch.nn.Parameter, torch.Tensor]] = {}
        self._alt: Dict[Tuple[int, str], Tuple[torch.nn.Parameter, torch.Tensor, object]] = {}
        self._slots: Dict[int, Tuple[int, torch.nn.Parameter]] = {}
        self._flat: Dict[torch.device, torch.Tensor] = {}
        if params is not None:
            sizes: Dict[torch.device, int] = {}
            for p in params:
                if not p.requires_grad or id(p) in self._slots:
                    continue
                off = sizes.get(p.device, 0)
                self._slots[id(p)] = (off, p)
                sizes[p.device] = off + (p.numel() + 7) // 8 * 8          # 32-byte aligned slots (float4 / TMA friendly)
            for dev, total in sizes.items():
                self._flat[dev] = torch.zeros(total, device=dev, dtype=torch.float32)

    def of(self, param: torch.Tensor) -> torch.Tensor:
        """Accumulation buffer with the parameter's shape."""
        hit = self._g.get(id(param))
        if hit is None:
            slot = self._slots.get(id(param))
            if slot is not None:
                buf = self._flat[param.device][slot[0]:slot[0] + param.numel()].view(param.shape)
            else:
                buf = torch.zeros(param.shape, device=param.device, dtype=torch.float32)
            hit = (param, buf)
            self._g[id(param)] = hit
        return hit[1]

    def _alt_buf(self, param, kind: str, shape, back) -> torch.Tensor:
        hit = self._alt.get((id(param), kind))
        if hit is None:
            hit = (param, torch.zeros(shape, device=param.device, dtype=torch.float32), back)
            self._alt[(id(param), kind)] = hit
        return hit[1]

    def table_t(self, param: torch.Tensor) -> torch.Tensor:
        """relative_position_bias_table is [L, nH]; the attention kernels work on its transpose [nH, L]."""
        return self._alt_buf(param, "table_t", (param.shape[1], param.shape[0]), lambda b: b.t())

    def conv_taps(self, param: torch.Tensor) -> torch.Tensor:
        """Conv2d / Conv3d weight [Cout, Cin, (kd,) kh, kw] accumulated tap-major [Cout, tap*Cin + ci] (the implicit-GEMM operand
        layout, tap = (kz*3 + ky)*3 + kx or ky*3 + kx)."""
        Cout, Cin = param.shape[:2]
        ks = tuple(param.shape[2:])
        taps = 1
        for k in ks:
            taps *= k
        nd = len(ks)
        perm = (0, nd + 1) + tuple(range(1, nd + 1))
        return self._alt_buf(param, "taps", (Cout, taps * Cin), lambda b: b.view(Cout, *ks, Cin).permute(*perm))

    def padded_cols(self, param: torch.Tensor, cols: int) -> torch.Tensor:
        """Weight flattened to [out, in] with the input axis zero-padded to ``cols`` (patch-embed GEMM, K = 48 -> 64)."""
        out = param.shape[0]
        kin = param.numel() // out
        return self._alt_buf(param, "pad%d" % cols, (out, cols), lambda b: b[:, :kin].reshape(param.shape))

    def _fold(self) -> None:
        for param, buf, back in self._alt.values():
            self.of(param).add_(back(buf))
        self._alt.clear()

    def finalize(self, only=None) -> List[torch.nn.Parameter]:
        """Hand the accumulated gradients to ``param.grad`` (added to an existing ``.grad`` like autograd does) and forget them.
        ``only``: restrict to these parameters (a finished stage whose gradients can already be all-reduced while the backward of
        the earlier stages runs).  Returns the parameters that received a gradient.  Tensor-container bookkeeping, not a hot path."""
        keep = None if only is None else {id(p) for p in only}
        done = []
        with torch.no_grad():
            for key in [k for k in self._alt if keep is None or k[0] in keep]:
                param, buf, back = self._alt.pop(key)
                self.of(param).add_(back(buf))
            for pid in [k for k in self._g if keep is None or k in keep]:
                param, buf = self._g.pop(pid)
                if not param.requires_grad:
                    continue
                g = buf.to(param.dtype)
                if param.grad is None:
                    param.grad = g
                else:
                    param.grad.add_(g)
                done.append(param)
        return done

    def flat_ranges(self, params) -> Tuple[List[torch.Tensor], List[torch.nn.Parameter]]:
        """Contiguous slices of the flat allocation that cover the slots of ``params`` (adjacent slots merged; the 32-byte slot padding
        between them holds zeros), plus the parameters that have no slot.  The gradient all-reduce runs IN PLACE on these slices --
        ``param.grad`` of a slotted fp32 parameter is a view of the same memory -- so no flatten / copy-back pass exists."""
        by_dev: Dict[torch.device, List[Tuple[int, int]]] = {}
        loose = []
        for p in params:
            slot = self._slots.get(id(p))
            if slot is None or p.dtype != torch.float32:
                loose.append(p)
                continue
            by_dev.setdefault(p.device, []).append((slot[0], slot[0] + (p.numel() + 7) // 8 * 8))
        views = []
        for dev, spans in by_dev.items():
            spans.sort()
            lo, hi = spans[0]
            for a, b in spans[1:]:
                if a <= hi:
                    hi = max(hi, b)
                else:
                    views.append(self._flat[dev][lo:hi])
                    lo, hi = a, b
            views.append(self._flat[dev][lo:hi])
        return views, loose

    def buffers(self) -> List[Tuple[torch.nn.Parameter, torch.Tensor]]:
        """(parameter, fp32 gradient buffer) pairs after folding the alternate layouts (gradient all-reduce, tests)."""
        with torch.no_grad():
            self._fold()
        return list(self._g.values())

    def named(self, module: torch.nn.Module) -> Dict[str, torch.Tensor]:
        """name -> gradient buffer for tests."""
        with torch.no_grad():
            self._fold()
        return {name: self._g[id(prm)][1] for name, prm in module.named_parameters() if id(prm) in self._g}


def _pad8(n: int) -> int:
    return (n + 7) // 8 * 8


def _transposed(ws: Workspace, name: str, x: torch.Tensor) -> torch.Tensor:
    """bf16 [M, N] -> workspace view [N, M8] (M8 = M rounded up to the 16-byte TMA pitch; pad columns zeroed)."""
    M, N = x.shape
    M8 = _pad8(M)
    buf = ws.get(name, (N, M8), torch.bfloat16, x.device)
    if M8 != M:
        buf[:, M:].zero_()
    K.transpose_bf16(x, buf[:, :M])
    return buf


def linear_bwd(dy: torch.Tensor, x: Optional[torch.Tensor], weight: torch.Tensor, bias: Optional[torch.Tensor], grads: GradStore,
               ws: Workspace, prepared: E.PreparedWeights, key: str, *, dx_bf16: Optional[torch.Tensor] = None,
               dx_f32: Optional[torch.Tensor] = None, dx_resid: Optional[torch.Tensor] = None, x_t: Optional[torch.Tensor] = None,
               bias_done: bool = False, **dx_epi) -> Optional[torch.Tensor]:
    """Adjoint of y = x W^T + b for bf16 rows dy [M, out], x [M, in]; ``weight`` is the [out, in(,1)] parameter.
    dW += dy^T x, db += colsum(dy); if a dx buffer is given: dx = dy W (through the GEMM epilogue options in ``dx_epi``).
    (``x_t`` is accepted for callers written against the transposed-operand version and ignored.)"""
    M, Nout = dy.shape
    w2 = weight.view(weight.shape[0], -1) if weight.dim() != 2 else weight
    Kin = w2.shape[1]
    dev = dy.device
    if weight.requires_grad:
        # dW += dy^T x straight from the row-major rows: 64-token x 64-channel TMA boxes are MN-major tcgen05 operands
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(Nout, Kin, M),), torch.float32, dev)
        K.gemm_bf16_wgrad(dy, x, grads.of(weight).view(Nout, Kin), part, accumulate=True)
        _count(2)
    if bias is not None and bias.requires_grad and not bias_done:      # (bias_done: the kernel that produced dy already summed its columns)
        K.colsum_accumulate(dy, grads.of(bias))
        _count(1)
    if dx_bf16 is not None or dx_f32 is not None:
        w_t = prepared.get(key + "_wT", [weight], lambda: _bf16(w2.t()))      # [in, out]
        K.gemm_bf16(dy, w_t, out_bf16=dx_bf16, out_f32=dx_f32, resid=dx_resid, **dx_epi)
        _count(1)
    return x_t


# ------------------------------------------------------------------------------------------------
# Swin block  (reference SwinTransformerBlock3D.forward, lib/video_swin_transformer.py:214-273)
# ------------------------------------------------------------------------------------------------
def draw_drop_path(rate: float, B: int, device) -> Optional[torch.Tensor]:
    """timm DropPath as the reference uses it (lib/video_swin_transformer.py:210, 266, 271): one Bernoulli(keep) draw per sample,
    scaled by 1 / keep.  Returns the fp32 [B] branch scale, or None when the rate is 0."""
    if rate <= 0.0:
        return None
    keep = 1.0 - rate
    return torch.empty(B, device=device, dtype=torch.float32).bernoulli_(keep).div_(keep)


# 0 (default): fc1 saves its pre-activation and the fc2 input-gradient epilogue evaluates GELU' of it; 1: fc1 saves GELU'(pre) in bf16 and
# the backward multiplies by it.  Same launches and the same time (148 us per stage-2 block for both GEMMs, 218 us with the two GELU
# kernels of the first version), but the bf16-rounded derivative moved one cancellation-heavy gradient (layers.0.blocks.0.norm1.bias)
# below the end-to-end direction criterion (cosine 0.934 < 0.95), so the derivative is evaluated in fp32 from the saved pre-activation.
_GELU_PRE_MODE = int(os.environ.get("LAVT_TRAIN_GELU_PRE_MODE", "0"))
# 1: the casts of a block's output gradient also sum its columns (d fc2.bias, d proj.bias; lavt_cast_rows_colsum_bf16), 48 launches fewer per
# step; 0 (default): separate column-sum launches.  Measured on one box, twice each: 65.5 / 65.8 ms fused vs 64.2 / 64.6 ms separate -- the
# column sums read the bf16 copy out of L2 right after the cast wrote it, and the fused kernel's register accumulators + per-block atomics cost
# more than that second pass, so the fusion stays an option.
_FUSE_COLSUM = int(os.environ.get("LAVT_TRAIN_FUSE_COLSUM", "0"))


def swin_block_fwd(x: torch.Tensor, blk, B: int, D: int, H: int, W: int, window, shifted: bool, clamp: bool, ws: Workspace,
                   xb_out: Optional[torch.Tensor] = None, drop_scales=None):
    """x fp32 [B*D*H*W, C] (not modified) -> (x_out, saved).  Same kernels as ``engine.swin_block`` except that fc1 also stores
    its pre-activation (second output of the same epilogue; ``hpre`` below) and nothing is overwritten.  ``drop_scales`` = (attention-branch scale,
    MLP-branch scale), fp32 [B] each or None (stochastic depth; drawn here from the block's rate when not given)."""
    n, C = x.shape
    dev = x.device
    geom = window_geometry(B, D, H, W, window, shifted, clamp)
    rows = geom.rows()
    nH = blk.num_heads
    pw = blk.prepared
    hd = C // nH
    qkv_w = pw.get("qkv_w", [blk.attn.qkv.weight], lambda: _bf16(blk.attn.qkv.weight))

    def _qscale():
        s = torch.ones(3 * C, device=dev, dtype=torch.float32)
        s[:C] = hd ** -0.5 * 1.4426950408889634
        b = _f32(blk.attn.qkv.bias) * s if blk.attn.qkv.bias is not None else torch.zeros(3 * C, device=dev)
        return s, b
    qkv_s, qkv_b = pw.get("qkv_sb", [blk.attn.qkv.weight] + ([blk.attn.qkv.bias] if blk.attn.qkv.bias is not None else []), _qscale)
    proj_w = pw.get("proj_w", [blk.attn.proj.weight], lambda: _bf16(blk.attn.proj.weight))
    fc1_w = pw.get("fc1_w", [blk.mlp.fc1.weight], lambda: _bf16(blk.mlp.fc1.weight))
    fc2_w = pw.get("fc2_w", [blk.mlp.fc2.weight], lambda: _bf16(blk.mlp.fc2.weight))
    table_t = pw.get("table_t", [blk.attn.relative_position_bias_table], lambda: _f32(blk.attn.relative_position_bias_table.t()))
    hidden = fc1_w.shape[0]
    if drop_scales is None:
        rate = float(getattr(blk, "drop_path_rate", 0.0)) if blk.training else 0.0
        drop_scales = (draw_drop_path(rate, B, dev), draw_drop_path(rate, B, dev))      # two independent draws, like the two DropPath calls
    s_attn, s_mlp = drop_scales
    tok = D * H * W

    xw = torch.empty(rows, C, device=dev, dtype=torch.bfloat16)
    K.layernorm_window_gather(x, geom, blk.norm1.weight, blk.norm1.bias, xw, eps=blk.norm1.eps)
    qkv = torch.empty(rows, 3 * C, device=dev, dtype=torch.bfloat16)
    K.gemm_bf16(xw, qkv_w, cscale=qkv_s, bias=qkv_b, out_bf16=qkv)
    att = torch.empty(rows, C, device=dev, dtype=torch.bfloat16)
    # row log-sum-exp of the scores, saved for the backward when the tcgen05 kernel runs (else the backward recomputes it)
    lse = torch.empty(rows, nH, device=dev, dtype=torch.float32) if K.window_attention_has_lse(table_t, geom) else None
    K.window_attention(qkv, table_t, geom, att, lse=lse)
    x1 = torch.empty_like(x)
    K.gemm_bf16(att, proj_w, bias=blk.attn.proj.bias.detach(), resid=x, out_f32=x1, win=geom, rscale=s_attn, rscale_rows=tok)
    h1 = torch.empty(n, C, device=dev, dtype=torch.bfloat16)
    K.layernorm_rows(x1, blk.norm2.weight, blk.norm2.bias, out_bf16=h1, eps=blk.norm2.eps)
    hpre = torch.empty(n, hidden, device=dev, dtype=torch.bfloat16)
    hid = torch.empty(n, hidden, device=dev, dtype=torch.bfloat16)
    # one epilogue writes GELU(pre) and the pre-activation (or GELU'(pre), see _GELU_PRE_MODE)
    K.gemm_bf16(h1, fc1_w, bias=blk.mlp.fc1.bias.detach(), act=K.ACT_GELU, out_bf16=hid, out_pre=hpre, pre_mode=_GELU_PRE_MODE)
    x2 = torch.empty_like(x)
    K.gemm_bf16(hid, fc2_w, bias=blk.mlp.fc2.bias.detach(), resid=x1, out_f32=x2, out_bf16=xb_out, rscale=s_mlp, rscale_rows=tok)
    _count(7)
    return x2, (x, xw, qkv, att, x1, h1, hpre, hid, geom, table_t, s_attn, s_mlp, tok, lse)


def swin_block_bwd(blk, saved, dx: torch.Tensor, grads: GradStore, ws: Workspace) -> torch.Tensor:
    """dx fp32 [n, C] = gradient of the block output; updated IN PLACE to the gradient of the block input and returned."""
    x0, xw, qkv, att, x1, h1, hpre, hid, geom, table_t, s_attn, s_mlp, tok, lse = saved
    n, C = x0.shape
    dev = x0.device
    rows = geom.rows()
    hidden = hid.shape[1]
    pw = blk.prepared
    # ---- MLP half: x2 = x1 + fc2(GELU(fc1(LN2(x1))))
    dyb = ws.get("bw_dyb", (n, C), torch.bfloat16, dev)
    # DropPath: the branch sees the gradient times its sample's scale; the same pass sums the columns = d fc2.bias
    b2 = blk.mlp.fc2.bias
    fuse2 = bool(_FUSE_COLSUM) and b2 is not None and b2.requires_grad and C <= 1024
    K.cast_rows_bf16(dx, dyb, rscale=s_mlp, rscale_rows=tok, colsum=grads.of(b2) if fuse2 else None)
    dhid = ws.get("bw_dhid", (n, hidden), torch.bfloat16, dev)
    # d pre = (dy W2) * GELU'(pre) in the epilogue of the input-gradient GEMM (`mul` operand = the saved pre-activation)
    linear_bwd(dyb, hid, blk.mlp.fc2.weight, blk.mlp.fc2.bias, grads, ws, pw, "fc2", dx_bf16=dhid, mul=hpre,
               mul_act=K.ACT_NONE if _GELU_PRE_MODE else K.ACT_GELU, bias_done=fuse2)
    dh1 = ws.get("bw_dh1", (n, C), torch.bfloat16, dev)
    linear_bwd(dhid, h1, blk.mlp.fc1.weight, blk.mlp.fc1.bias, grads, ws, pw, "fc1", dx_bf16=dh1)
    K.layernorm_rows_bwd(x1, dh1, blk.norm2.weight, dx, grads.of(blk.norm2.weight), grads.of(blk.norm2.bias), dres=dx,
                         eps=blk.norm2.eps)
    # ---- attention half: x1 = x0 + scatter(proj(attn(qkv(gather(LN1(x0))))))
    dyw = ws.get("bw_dyw", (rows, C), torch.bfloat16, dev)
    bp = blk.attn.proj.bias
    fusep = bool(_FUSE_COLSUM) and bp is not None and bp.requires_grad and C <= 1024
    K.cast_rows_bf16(dx, dyw, geom, rscale=s_attn, rscale_rows=tok, colsum=grads.of(bp) if fusep else None)
    datt = ws.get("bw_datt", (rows, C), torch.bfloat16, dev)
    linear_bwd(dyw, att, blk.attn.proj.weight, blk.attn.proj.bias, grads, ws, pw, "proj", dx_bf16=datt, bias_done=fusep)
    dqkv = ws.get("bw_dqkv", (rows, 3 * C), torch.bfloat16, dev)
    tbl = blk.attn.relative_position_bias_table
    nws = K.window_attention_bwd_workspace_floats(table_t, geom) if lse is not None else 0
    aws = ws.get("bw_attn", (nws,), torch.float32, dev) if nws > 0 else None
    K.window_attention_bwd(qkv, att, datt, table_t, geom, dqkv, grads.table_t(tbl) if tbl.requires_grad else None, lse=lse, workspace=aws)
    dxw = ws.get("bw_dxw", (rows, C), torch.bfloat16, dev)
    linear_bwd(dqkv, xw, blk.attn.qkv.weight, blk.attn.qkv.bias, grads, ws, pw, "qkv", dx_bf16=dxw)
    K.layernorm_window_gather_bwd(x0, geom, dxw, blk.norm1.weight, dx, grads.of(blk.norm1.weight), grads.of(blk.norm1.bias),
                                  dres=dx, eps=blk.norm1.eps)
    _count(6)
    return dx


# ------------------------------------------------------------------------------------------------
# PatchMerging (reference :289-311)
# ------------------------------------------------------------------------------------------------
def patch_merging_fwd(x: torch.Tensor, ds, B: int, D: int, H: int, W: int, ws: Workspace):
    C = x.shape[1]
    dev = x.device
    H2, W2 = (H + 1) // 2, (W + 1) // 2
    red_w = ds.prepared.get("red_w", [ds.reduction.weight], lambda: _bf16(ds.reduction.weight))
    g = torch.empty(B * D * H2 * W2, 4 * C, device=dev, dtype=torch.bfloat16)
    K.patch_merge_layernorm(x, B, D, H, W, ds.norm.weight, ds.norm.bias, g, eps=ds.norm.eps)
    out = torch.empty(B * D * H2 * W2, 2 * C, device=dev, dtype=torch.float32)
    K.gemm_bf16(g, red_w, out_f32=out)
    _count(2)
    return out, (x, g, (B, D, H, W))


def patch_merging_bwd(ds, saved, dout: torch.Tensor, grads: GradStore, ws: Workspace) -> torch.Tensor:
    """dout fp32 [rows/4, 2C] -> dx fp32 [rows, C] (new tensor)."""
    x, g, (B, D, H, W) = saved
    dev = x.device
    C = x.shape[1]
    dyb = ws.get("bw_dyb2", tuple(dout.shape), torch.bfloat16, dev)
    K.cast_rows_bf16(dout, dyb)
    dg = ws.get("bw_dmerge", tuple(g.shape), torch.bfloat16, dev)
    linear_bwd(dyb, g, ds.reduction.weight, None, grads, ws, ds.prepared, "red", dx_bf16=dg)
    dx = torch.empty_like(x)
    if (H % 2) or (W % 2):
        pass    # every real token still belongs to exactly one merged row; padded positions have no source token
    K.patch_merge_layernorm_bwd(x, B, D, H, W, dg, ds.norm.weight, dx, grads.of(ds.norm.weight), grads.of(ds.norm.bias), eps=ds.norm.eps)
    _count(2)
    return dx


# ------------------------------------------------------------------------------------------------
# PWAM + LanguageGate  (reference PWAM.forward :919-934, SpatialImageLanguageAttention.forward :975-1009, res_gate :519-525)
# ------------------------------------------------------------------------------------------------
def _nl_pad(Nl: int) -> int:
    return (Nl + 7) // 8 * 8


def _att_ln_bwd(x_raw: torch.Tensor, dy: torch.Tensor, ln, grads: GradStore, ws: Workspace, name: str) -> torch.Tensor:
    """Adjoint of the row LayerNorm that --att_norm_layer_type LN puts behind f_query / W: x_raw fp32 [B,n,C] = its input, dy bf16 [B*n, C] =
    gradient of its output -> bf16 gradient of its input (LayerNorm backward kernel + the bf16 cast the next weight-gradient GEMM reads)."""
    N_, C = dy.shape
    dev = dy.device
    dx32 = ws.get(name + "_f32", (N_, C), torch.float32, dev)
    K.layernorm_rows_bwd(x_raw.view(N_, C), dy, ln.weight, dx32, grads.of(ln.weight), grads.of(ln.bias), eps=ln.eps)
    out = ws.get(name + "_bf16", (N_, C), torch.bfloat16, dev)
    K.cast_rows_bf16(dx32, out)
    _count(2)
    return out


def _att_bn_fwd(raw: torch.Tensor, bn, B: int, ws: Workspace):
    """--att_norm_layer_type BN in training mode (nn.BatchNorm1d in train(), reference lib/backbone.py:1297-1316): batch statistics over all
    clips and tokens of ``raw`` fp32 [B,n,C].  Nothing is materialised: the affine normalisation y = (x - mean) rstd gamma + beta is handed to
    the consumers as FOLDED statistics (mean' = mean - beta / (rstd gamma), rstd' = rstd gamma), which they already apply per element.
    Returns (folded statistics [B,2,C], true statistics [2,C])."""
    Bq, n, C = raw.shape
    dev = raw.device
    if _world() is not None:
        raise NotImplementedError("--att_norm_layer_type BN under SyncBatchNorm (multi-GPU training) is not implemented on the B200 path")
    N_ = Bq * n
    stats = torch.empty(1, 2, C, device=dev, dtype=torch.float32)
    stw = ws.get("pw_statw1", (K.instnorm_workspace_floats(1, N_, C),), torch.float32, dev)
    K.instnorm_stats(raw.view(1, N_, C), stats, stw, eps=bn.eps)
    _count(2)
    with torch.no_grad():       # [C]-sized bookkeeping: folded statistics and the running buffers
        mean, rstd = stats[0, 0], stats[0, 1]
        if bn.track_running_stats:
            mom = bn.momentum if bn.momentum is not None else 0.1
            var = 1.0 / rstd ** 2 - bn.eps
            bn.running_mean.mul_(1 - mom).add_(mean, alpha=mom)
            bn.running_var.mul_(1 - mom).add_(var * (N_ / max(N_ - 1, 1)), alpha=mom)
            bn.num_batches_tracked += 1
        gam = bn.weight.detach().float()
        gam = torch.where(gam.abs() < 1e-12, torch.full_like(gam, 1e-12), gam)
        rs2 = rstd * gam
        folded = torch.stack([mean - bn.bias.detach().float() / rs2, rs2]).unsqueeze(0).expand(B, 2, C).contiguous()
    return folded, stats.view(2, C)


def _att_bn_bwd(raw: torch.Tensor, stats: torch.Tensor, g: torch.Tensor, bn, grads: GradStore, ws: Workspace, pw, name: str) -> torch.Tensor:
    """Adjoint of the BatchNorm above: raw fp32 [B,n,C], true statistics [2,C], g bf16 [B*n, C] = gradient of the BatchNorm output.
    The decoder's BatchNorm + ReLU adjoint kernels are reused with an all-ones ReLU mask.  Returns the bf16 gradient of ``raw``."""
    N_, C = g.shape
    dev = g.device
    ones = pw.get("bn_ones_%d_%d" % (N_, C), [], lambda: torch.ones(N_, C, device=dev, dtype=torch.bfloat16))
    sums = torch.zeros(2, C, device=dev, dtype=torch.float32)
    z = raw.view(N_, C)
    K.bn_relu_bwd_reduce(g, ones, z, stats, sums)
    with torch.no_grad():
        if bn.weight.requires_grad:
            grads.of(bn.weight).add_(sums[1])
        if bn.bias.requires_grad:
            grads.of(bn.bias).add_(sums[0])
    out = ws.get(name, (N_, C), torch.bfloat16, dev)
    K.bn_relu_bwd_apply(g, ones, z, stats, bn.weight, sums, out, N_)
    _count(2)
    return out


def _mm_and_gate_fwd(x, a2, fusion, res_gate, mm_w, gate_act):
    """r = GELU(project_mm(a2)) (:930) and the LanguageGate (:519-525) with what their adjoints need."""
    N_, C = x.shape
    dev = x.device
    pw = fusion.prepared
    bf, f32 = torch.bfloat16, torch.float32
    rpre = torch.empty(N_, C, device=dev, dtype=bf)
    K.gemm_bf16(a2.view(N_, C), mm_w, bias=fusion.project_mm[0].bias.detach(), out_bf16=rpre)
    rb = torch.empty(N_, C, device=dev, dtype=bf)
    r32 = torch.empty(N_, C, device=dev, dtype=f32)
    K.gate_elementwise(3, rpre, out_bf16=rb, out_f32=r32)
    _count(12)
    g1 = g2 = xg = None
    if res_gate is not None:
        g0w = pw.get("g0", [res_gate[0].weight], lambda: _bf16(res_gate[0].weight))
        g2w = pw.get("g2", [res_gate[2].weight], lambda: _bf16(res_gate[2].weight))
        g1 = torch.empty(N_, C, device=dev, dtype=bf)
        K.gemm_bf16(rb, g0w, act=K.ACT_RELU, out_bf16=g1)
        g2 = torch.empty(N_, C, device=dev, dtype=bf)
        K.gemm_bf16(g1, g2w, out_bf16=g2)       # PRE-activation of the tanh / sigmoid (saved); the gate is applied by the elementwise kernel
        xg = torch.empty(N_, C, device=dev, dtype=f32)
        K.gate_elementwise(0 if gate_act == "tanh" else 7, g2, rb, f=x, out_f32=xg)
        _count(3)
    return rpre, rb, r32, g1, g2, xg


def _simple_fuse_fwd(x, xb, fusion, res_gate, l, mask, B, ws, gate_act, vispre, vis, mm_w):
    """--fuse simple in training mode: a2 = vis * LangProject(l) (one sentence vector per clip, reference :916-917, :929-930, :1012-1039).
    The sentence vector sits in an InstanceNorm-statistics block as (mean = -s, rstd = 1) over an all-zero lang_pre tensor, so the PWAM
    product kernel and ITS ADJOINT are reused: row 0 of the adjoint's reductions is sum_pixels d a2 * vis = d s."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    pr = fusion.image_lang_att.project
    stats = torch.empty(B, 2, C, device=dev, dtype=torch.float32)
    K.lang_project(l, mask, _f32(pr[0].weight), _f32(pr[0].bias), _f32(pr[2].weight), _f32(pr[2].bias), stats)
    zeros = pw.get("zeros_%d_%d" % (B, n), [], lambda: torch.zeros(B, n, C, device=dev, dtype=torch.float32))
    a2 = torch.empty(B, n, C, device=dev, dtype=torch.bfloat16)
    K.pwam_mul_norm(vis, zeros, stats, a2)
    rpre, rb, r32, g1, g2, xg = _mm_and_gate_fwd(x, a2, fusion, res_gate, mm_w, gate_act)
    saved = dict(xb=xb, vispre=vispre, vis=vis, langpre=zeros, stats_l=stats, a2=a2, rpre=rpre, rb=rb, g1=g1, g2=g2, l=l, mask=mask, B=B,
                 heads=1, gate_act=gate_act, no_norm=False, simple=True)
    return r32, xg, saved


def pwam_gate_fwd(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, ws: Workspace,
                  gate_act: str = "tanh"):
    """x fp32 [B*n, C] (not modified), xb = its bf16 copy, l fp32 [B,768,Nl], mask fp32 [B,Nl].
    Returns (r fp32 [B*n, C] = x_residual, x' fp32 = gated x or None without a gate, saved)."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    att = fusion.image_lang_att
    heads = getattr(att, "num_heads", 1)
    Nl = l.shape[-1]
    bf, f32 = torch.bfloat16, torch.float32

    def wprep(name, conv):
        return pw.get(name, [conv.weight], lambda: _bf16(conv.weight[:, :, 0]))
    simple = not fusion.attention          # --fuse simple (reference :916-917, :929-930): lang = LangProject(mean-pooled words), one vector per clip
    vis_w, mm_w = wprep("vis_w", fusion.vis_project[0]), wprep("mm_w", fusion.project_mm[0])
    if not simple:
        q_w, W_w = wprep("q_w", att.f_query[0]), wprep("W_w", att.W[0])
        k_w = pw.get("k_w", [att.f_key[0].weight], lambda: _f32(att.f_key[0].weight[:, :, 0]))
        v_w = pw.get("v_w", [att.f_value[0].weight], lambda: _f32(att.f_value[0].weight[:, :, 0]))
    else:
        k_w = v_w = None

    vispre = torch.empty(N_, C, device=dev, dtype=bf)
    vis = torch.empty(B, n, C, device=dev, dtype=bf)
    K.gemm_bf16(xb, vis_w, bias=fusion.vis_project[0].bias.detach(), act=K.ACT_GELU, out_bf16=vis.view(N_, C), out_pre=vispre)
    if simple:
        return _simple_fuse_fwd(x, xb, fusion, res_gate, l, mask, B, ws, gate_act, vispre, vis, mm_w)
    qpre = torch.empty(B, n, C, device=dev, dtype=f32)
    K.gemm_bf16(xb, q_w, bias=att.f_query[0].bias.detach(), out_f32=qpre.view(N_, C))
    # --att_norm_layer_type none / LN (2-D backbone, reference lib/backbone.py:1297-1316): Identity or a row LayerNorm instead of
    # InstanceNorm1d -- the consumers read identity "statistics" (mean 0, rstd 1) of the (LayerNorm'd) projection and the backward's
    # InstanceNorm reductions are zeroed, which turns its adjoint into a pass-through; LN adds the LayerNorm adjoint behind it
    norm_kind = getattr(att, "att_norm_layer_type", "IN")
    if norm_kind not in ("IN", "none", "LN", "BN"):
        raise NotImplementedError("--att_norm_layer_type %s is not known" % norm_kind)
    ident = None
    q_raw = l_raw = None
    bn_q = bn_l = None            # BN: (folded statistics [B,2,C], true statistics [2,C])
    if norm_kind != "IN":
        ident = pw.get("ident_%d_%s" % (B, dev), [], lambda: torch.stack([torch.zeros(B, C), torch.ones(B, C)], 1).to(dev).contiguous())
    if norm_kind == "LN":
        q_raw = qpre                                            # LayerNorm input, kept for its adjoint
        qpre = torch.empty(B, n, C, device=dev, dtype=f32)
        K.layernorm_rows(q_raw.view(N_, C), att.f_query[1].weight, att.f_query[1].bias, out_f32=qpre.view(N_, C), eps=att.f_query[1].eps)
        _count(1)
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(B, n, C),), f32, dev)
    if norm_kind == "BN":
        bn_q = _att_bn_fwd(qpre, att.f_query[1], B, ws)
        stats_q = bn_q[0]
    elif ident is None:
        stats_q = torch.empty(B, 2, C, device=dev, dtype=f32)
        K.instnorm_stats(qpre, stats_q, stw)
    else:
        stats_q = ident
    kk = torch.empty(B, Nl, C, device=dev, dtype=f32)
    vv = torch.empty(B, Nl, C, device=dev, dtype=f32)
    K.pwam_kv(l, mask, k_w, att.f_key[0].bias.detach(), v_w, att.f_value[0].bias.detach(), kk, vv)
    o = torch.empty(B, n, C, device=dev, dtype=bf)
    K.pwam_attend(qpre, stats_q, kk, vv, mask, o, heads)
    langpre = torch.empty(B, n, C, device=dev, dtype=f32)
    K.gemm_bf16(o.view(N_, C), W_w, bias=att.W[0].bias.detach(), out_f32=langpre.view(N_, C))
    if norm_kind == "LN":
        l_raw = langpre
        langpre = torch.empty(B, n, C, device=dev, dtype=f32)
        K.layernorm_rows(l_raw.view(N_, C), att.W[1].weight, att.W[1].bias, out_f32=langpre.view(N_, C), eps=att.W[1].eps)
        _count(1)
    if norm_kind == "BN":
        bn_l = _att_bn_fwd(langpre, att.W[1], B, ws)
        stats_l = bn_l[0]
    elif ident is None:
        stats_l = torch.empty(B, 2, C, device=dev, dtype=f32)
        K.instnorm_stats(langpre, stats_l, stw)
    else:
        stats_l = ident
    a2 = torch.empty(B, n, C, device=dev, dtype=bf)
    K.pwam_mul_norm(vis, langpre, stats_l, a2)
    rpre, rb, r32, g1, g2, xg = _mm_and_gate_fwd(x, a2, fusion, res_gate, mm_w, gate_act)
    saved = dict(xb=xb, vispre=vispre, vis=vis, qpre=qpre, stats_q=stats_q, kk=kk, vv=vv, o=o, langpre=langpre, stats_l=stats_l,
                 a2=a2, rpre=rpre, rb=rb, g1=g1, g2=g2, l=l, mask=mask, B=B, heads=heads, k_w=k_w, v_w=v_w, gate_act=gate_act,
                 no_norm=ident is not None, simple=False, q_raw=q_raw, l_raw=l_raw, bn_q=bn_q, bn_l=bn_l, ident=ident)
    return r32, xg, saved


def pwam_gate_bwd(fusion, res_gate, saved, dr_out: Optional[torch.Tensor], dxg: Optional[torch.Tensor], grads: GradStore, ws: Workspace,
                  dl: torch.Tensor) -> torch.Tensor:
    """dr_out fp32 [B*n, C]: gradient of r from the stage-output path (or None); dxg fp32: gradient of the gated x' (or None when the
    gate output is unused, e.g. the last stage).  ``dl`` fp32 [B,768,Nl] accumulates the gradient of the language features.
    Returns dx fp32 [B*n, C], the gradient of the stage features x (dxg is reused in place when given)."""
    s = saved
    B, heads = s["B"], s["heads"]
    xb = s["xb"]
    N_, C = xb.shape
    n = N_ // B
    dev = xb.device
    bf, f32 = torch.bfloat16, torch.float32
    pw = fusion.prepared
    att = fusion.image_lang_att
    Nl = s["l"].shape[-1]
    nlp = _nl_pad(Nl)
    dr = dr_out
    if res_gate is not None and dxg is not None:
        dg2pre = ws.get("bw_pw_a", (N_, C), bf, dev)
        gmode = 1 if s.get("gate_act", "tanh") == "tanh" else 8
        if dr is None:
            dr = ws.get("bw_pw_dr", (N_, C), f32, dev)
            K.gate_elementwise(gmode, s["g2"], s["rb"], f=dxg, f2=None, out_bf16=dg2pre, out_f32=dr)
        else:
            K.gate_elementwise(gmode, s["g2"], s["rb"], f=dxg, f2=dr, out_bf16=dg2pre, out_f32=dr)
        dg1 = ws.get("bw_pw_b", (N_, C), bf, dev)
        linear_bwd(dg2pre, s["g1"], res_gate[2].weight, None, grads, ws, pw, "g2", dx_bf16=dg1)
        K.gate_elementwise(2, dg1, s["g1"], out_bf16=dg1)
        linear_bwd(dg1, s["rb"], res_gate[0].weight, None, grads, ws, pw, "g0", dx_f32=dr, dx_resid=dr)
        _count(2)
    if dr is None:
        raise K.LavtError("pwam backward: neither the stage output nor the gated features carry a gradient")
    drpre = ws.get("bw_pw_a", (N_, C), bf, dev)
    K.gate_elementwise(4, s["rpre"], f=dr, out_bf16=drpre)
    da2 = ws.get("bw_pw_b", (N_, C), bf, dev)
    linear_bwd(drpre, s["a2"].view(N_, C), fusion.project_mm[0].weight, fusion.project_mm[0].bias, grads, ws, pw, "mm", dx_bf16=da2)
    sums = torch.zeros(2, B, 2, C, device=dev, dtype=f32)
    dvispre = ws.get("bw_pw_c", (N_, C), bf, dev)
    K.pwam_mul_norm_bwd(da2, s["vis"], s["vispre"], s["langpre"], s["stats_l"], dvispre, sums[0])
    if s.get("simple"):
        # --fuse simple: d s = sum_pixels d a2 * vis (row 0 of the reductions) -> LangProject adjoint; the only projection of x is vis_project
        pr = att.project
        ds = sums[0][:, 0, :].contiguous()
        Lin = s["l"].shape[1]
        wsp = ws.get("bw_langproj", (B * (2 * C + 2 * Lin),), f32, dev)

        def gof(prm):
            return grads.of(prm) if prm.requires_grad else None
        K.lang_project_bwd(s["l"], s["mask"], _f32(pr[0].weight), _f32(pr[0].bias), _f32(pr[2].weight), ds, gof(pr[0].weight), gof(pr[0].bias),
                           gof(pr[2].weight), gof(pr[2].bias), dl, wsp)
        if dxg is not None:
            dx, first_resid = dxg, dxg
        else:
            dx, first_resid = torch.empty(N_, C, device=dev, dtype=f32), None
        linear_bwd(dvispre, xb, fusion.vis_project[0].weight, fusion.vis_project[0].bias, grads, ws, pw, "vis", dx_f32=dx, dx_resid=first_resid)
        _count(12)
        return dx
    if s.get("no_norm"):
        sums[0].zero_()         # Identity instead of InstanceNorm: with zero reductions and rstd = 1 the adjoint below is the pass-through
    dlangpre = ws.get("bw_pw_a", (N_, C), bf, dev)
    # (BN: the kernels above normalised with the FOLDED statistics; the gradient of the BatchNorm OUTPUT is the pass-through of g = d a2 * vis)
    K.instnorm_bwd(s["langpre"], s["ident"] if s.get("bn_l") is not None else s["stats_l"], sums[0], dlangpre, ga=da2, gb=s["vis"].view(N_, C))
    if s.get("bn_l") is not None:
        dlangpre = _att_bn_bwd(s["langpre"], s["bn_l"][1], dlangpre, att.W[1], grads, ws, pw, "bw_pw_bn")
    if s.get("l_raw") is not None:          # --att_norm_layer_type LN: dlangpre is the gradient of the LayerNorm OUTPUT
        dlangpre = _att_ln_bwd(s["l_raw"], dlangpre, att.W[1], grads, ws, "bw_pw_ln")
    do = ws.get("bw_pw_b", (N_, C), bf, dev)
    linear_bwd(dlangpre, s["o"].view(N_, C), att.W[0].weight, att.W[0].bias, grads, ws, pw, "W", dx_bf16=do)
    # pixel-word attention core
    Wd = B * heads * nlp
    dqhat = ws.get("bw_pw_dq", (B, n, C), f32, dev)
    qs = ws.get("bw_pw_a", (N_, C), bf, dev)
    p_bd = ws.get("bw_pw_pbd", (N_, Wd), bf, dev)
    ds_bd = ws.get("bw_pw_dsbd", (N_, Wd), bf, dev)
    K.pwam_attend_bwd(s["qpre"], s["stats_q"], s["kk"], s["vv"], s["mask"], do, dqhat, qs, p_bd, ds_bd, sums[1], heads, nlp)
    dkv = torch.empty(2, Wd, C, device=dev, dtype=f32)
    for buf, dy_rows, x_rows in ((dkv[0], ds_bd, qs), (dkv[1], p_bd, do)):      # dk = dS^T (C^-0.5 q^), dv = P^T dO
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(Wd, C, N_),), f32, dev)
        K.gemm_bf16_wgrad(dy_rows, x_rows, buf, part, accumulate=False)
    fk, fv = att.f_key[0], att.f_value[0]
    K.pwam_kv_bwd(dkv[0], dkv[1], s["mask"], s["l"], s["k_w"], s["v_w"],
                  grads.of(fk.weight) if fk.weight.requires_grad else None, grads.of(fk.bias) if fk.bias.requires_grad else None,
                  grads.of(fv.weight) if fv.weight.requires_grad else None, grads.of(fv.bias) if fv.bias.requires_grad else None,
                  dl, heads, nlp)
    if s.get("no_norm"):
        sums[1].zero_()
    dqpre = ws.get("bw_pw_b", (N_, C), bf, dev)
    K.instnorm_bwd(s["qpre"], s["ident"] if s.get("bn_q") is not None else s["stats_q"], sums[1], dqpre, g_f32=dqhat)
    if s.get("bn_q") is not None:
        dqpre = _att_bn_bwd(s["qpre"], s["bn_q"][1], dqpre, att.f_query[1], grads, ws, pw, "bw_pw_bn")
    if s.get("q_raw") is not None:
        dqpre = _att_ln_bwd(s["q_raw"], dqpre, att.f_query[1], grads, ws, "bw_pw_ln")
    # both projections of x: dx (+)= dvispre Wvis + dqpre Wq
    if dxg is not None:
        dx = dxg
        first_resid = dx
    else:
        dx = torch.empty(N_, C, device=dev, dtype=f32)
        first_resid = None
    x_t = linear_bwd(dvispre, xb, fusion.vis_project[0].weight, fusion.vis_project[0].bias, grads, ws, pw, "vis", dx_f32=dx,
                     dx_resid=first_resid)
    linear_bwd(dqpre, xb, att.f_query[0].weight, att.f_query[0].bias, grads, ws, pw, "q", dx_f32=dx, dx_resid=dx, x_t=x_t)
    _count(16)
    return dx


# ------------------------------------------------------------------------------------------------
# PatchEmbed3D (reference :616-634) and the per-stage output norm (:869-874)
# ------------------------------------------------------------------------------------------------
def patch_embed_fwd(x5: torch.Tensor, pe, ws: Workspace):
    """x5 fp32 (B,3,T,H,W) strided view -> (x fp32 [B*T*Hp*Wp, C], Hp, Wp, saved)."""
    B, _, T, H, W = x5.shape
    dev = x5.device
    Hp, Wp = (H + 3) // 4, (W + 3) // 4
    C = pe.embed_dim
    n = B * T * Hp * Wp

    def _w():
        w = pe.proj.weight.detach().reshape(C, -1).to(torch.bfloat16)
        wp = torch.zeros(C, 64, device=w.device, dtype=torch.bfloat16)
        wp[:, : w.shape[1]] = w
        return wp
    pw_ = pe.prepared.get("w", [pe.proj.weight], _w)
    cols = torch.empty(n, 64, device=dev, dtype=torch.bfloat16)
    K.patch_embed_im2col(x5, cols)
    ypre = torch.empty(n, C, device=dev, dtype=torch.float32)
    K.gemm_bf16(cols, pw_, bias=pe.proj.bias.detach(), out_f32=ypre)
    if pe.norm is None:
        _count(2)
        return ypre, Hp, Wp, (cols, None)
    x = torch.empty(n, C, device=dev, dtype=torch.float32)
    K.layernorm_rows(ypre, pe.norm.weight, pe.norm.bias, out_f32=x, eps=pe.norm.eps)
    _count(3)
    return x, Hp, Wp, (cols, ypre)


def patch_embed_bwd(pe, saved, dx: torch.Tensor, grads: GradStore, ws: Workspace) -> None:
    """dx fp32 [n, C]: gradient of the patch-embedding output (the pixels need no gradient)."""
    cols, ypre = saved
    if not any(p.requires_grad for p in pe.parameters()):
        return
    n, C = dx.shape
    dev = dx.device
    dyb = ws.get("bw_dyb", (n, C), torch.bfloat16, dev)
    K.cast_rows_bf16(dx, dyb)
    if ypre is not None:
        dpre = ws.get("bw_pe_dpre", (n, C), torch.float32, dev)
        K.layernorm_rows_bwd(ypre, dyb, pe.norm.weight, dpre, grads.of(pe.norm.weight), grads.of(pe.norm.bias), eps=pe.norm.eps)
        K.cast_rows_bf16(dpre, dyb)
        _count(2)
    if pe.proj.weight.requires_grad:
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(C, 64, n),), torch.float32, dev)
        K.gemm_bf16_wgrad(dyb, cols, grads.padded_cols(pe.proj.weight, 64), part, accumulate=True)
        _count(2)
    if pe.proj.bias is not None and pe.proj.bias.requires_grad:
        K.colsum_accumulate(dyb, grads.of(pe.proj.bias))
        _count(1)
    _count(1)


# ------------------------------------------------------------------------------------------------
# SimpleDecoding in training mode (reference lib/mask_predictor.py:56-99, BatchNorm2d batch statistics / SyncBatchNorm train.py:589)
# ------------------------------------------------------------------------------------------------
def _world():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) else None


def _cbr_fwd(x_nhwc: torch.Tensor, dec, conv_name: str, bn_name: str, ws: Workspace, sync_bn: bool):
    conv, bn = getattr(dec, conv_name), getattr(dec, bn_name)
    n, H, W, Cin = x_nhwc.shape
    dev = x_nhwc.device
    hid = conv.weight.shape[0]
    npix = n * H * W
    w = dec.prepared.get(conv_name, [conv.weight], lambda: E._conv_taps(conv))
    z = torch.empty(npix, hid, device=dev, dtype=torch.float32)
    K.conv3x3_bf16(x_nhwc, w, out_f32=z)
    stats = torch.empty(1, 2, hid, device=dev, dtype=torch.float32)
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(1, npix, hid),), torch.float32, dev)
    K.instnorm_stats(z.view(1, npix, hid), stats, stw, eps=bn.eps)
    n_stat = npix
    dist = _world() if sync_bn else None
    with torch.no_grad():       # [C]-sized bookkeeping: cross-GPU statistics and the running buffers
        if dist is not None:
            mean = stats[0, 0]
            ex2 = 1.0 / stats[0, 1] ** 2 - bn.eps + mean * mean
            both = torch.stack([mean, ex2])
            dist.all_reduce(both)
            both /= dist.get_world_size()
            n_stat = npix * dist.get_world_size()
            stats[0, 0] = both[0]
            stats[0, 1] = torch.rsqrt((both[1] - both[0] * both[0]).clamp_min(0) + bn.eps)
        if bn.track_running_stats:
            mom = bn.momentum if bn.momentum is not None else 0.1
            var = 1.0 / stats[0, 1] ** 2 - bn.eps
            bn.running_mean.mul_(1 - mom).add_(stats[0, 0], alpha=mom)
            bn.running_var.mul_(1 - mom).add_(var * (n_stat / max(n_stat - 1, 1)), alpha=mom)
            bn.num_batches_tracked += 1
    t = torch.empty(n, H, W, hid, device=dev, dtype=torch.bfloat16)
    K.bn_relu_apply(z, stats.view(2, hid), bn.weight, bn.bias, t.view(npix, hid))
    _count(4)
    return t, (x_nhwc, z, stats.view(2, hid), t, n_stat, conv_name, bn_name)


def _cbr_bwd(dec, saved, dt: torch.Tensor, grads: GradStore, ws: Workspace, sync_bn: bool, dx_out: Optional[torch.Tensor]) -> None:
    """dt bf16 [npix, hid] = gradient of the ReLU output; writes the input gradient (bf16 NHWC) into ``dx_out`` if given."""
    x_nhwc, z, stats, t, n_stat, conv_name, bn_name = saved
    conv, bn = getattr(dec, conv_name), getattr(dec, bn_name)
    n, H, W, Cin = x_nhwc.shape
    dev = z.device
    npix, hid = z.shape
    sums = torch.zeros(2, hid, device=dev, dtype=torch.float32)
    K.bn_relu_bwd_reduce(dt, t.view(npix, hid), z, stats, sums)
    with torch.no_grad():
        dist = _world() if sync_bn else None
        if dist is not None:
            dist.all_reduce(sums)
        if bn.weight.requires_grad:
            grads.of(bn.weight).add_(sums[1])       # note: with SyncBN every rank holds the GLOBAL sum; the later gradient
        if bn.bias.requires_grad:                   # all-reduce averages, which reproduces SyncBatchNorm's DDP semantics
            grads.of(bn.bias).add_(sums[0])
    dz = ws.get("bw_dz", (n, H, W, hid), torch.bfloat16, dev)
    K.bn_relu_bwd_apply(dt, t.view(npix, hid), z, stats, bn.weight, sums, dz.view(npix, hid), n_stat)
    _count(2)
    if conv.weight.requires_grad and Cin % 64 == 0:
        # one launch: dz and x are read in place through 4-D TMA boxes (64 channels x 64 pixels = MN-major tcgen05 operands), the tap
        # is a coordinate offset of the x box, the zero padding TMA's out-of-bounds fill
        part = ws.get("bw_splitk", (K.conv3x3_wgrad_workspace_floats(n, H, W, Cin, hid),), torch.float32, dev)
        K.conv3x3_wgrad(dz, x_nhwc, grads.conv_taps(conv.weight), part, accumulate=True)
        _count(2)
    elif conv.weight.requires_grad:
        # channel counts that are not a multiple of 64 (Swin-T/S decoders): nine split-K GEMMs over zero-padded transposed layouts.
        # dW[co, tap, ci] = sum_p dz^T[co, p] x^T[ci, p + (ky-1)*Wp + (kx-1)] over the padded pixel axis (rows of Wp = W+2 rounded
        # up to 8 columns): the row part of the offset is a 16-byte aligned TMA coordinate, the +-1 part a pre-shifted copy of x^T
        Wp = _pad8(W + 2)
        Kp = n * (H + 2) * Wp
        dz_t = ws.get("bw_dzT", (hid, Kp), torch.bfloat16, dev)
        dz_t.zero_()
        K.nhwc_pad_transpose(dz, dz_t, Wp, 0)
        x_t = ws.get("bw_cxT", (3, Cin, Kp), torch.bfloat16, dev)
        x_t.zero_()
        for kx in range(3):
            K.nhwc_pad_transpose(x_nhwc, x_t[kx], Wp, kx - 1)
        gbuf = grads.conv_taps(conv.weight)
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(hid, Cin, Kp),), torch.float32, dev)
        for tap in range(9):
            ky, kx = tap // 3, tap % 3
            K.gemm_bf16_splitk(dz_t, x_t[kx], gbuf[:, tap * Cin:(tap + 1) * Cin], part, accumulate=True, b_koff=(ky - 1) * Wp)
        _count(6 + 18)
    if dx_out is not None:
        def _wT():
            wgt = conv.weight.detach()                         # [Cout, Cin, 3, 3] -> [Cin, ((2-ky)*3 + (2-kx))*Cout + co]
            return wgt.flip(2, 3).permute(1, 2, 3, 0).reshape(wgt.shape[1], -1).to(torch.bfloat16).contiguous()
        w_t = dec.prepared.get(conv_name + "_wT", [conv.weight], _wT)
        K.conv3x3_bf16(dz, w_t, out_bf16=dx_out.view(npix, Cin))
        _count(1)


def decoder_fwd(dec, c4, c3, c2, c1, ws: Workspace, sync_bn: bool = False):
    """NHWC bf16 maps (coarse -> fine) -> (low-resolution logits fp32 [n, H1, W1, 2], saved).  ``c1`` is None under --lazy_pred: the
    decoder stops at the 1/8-scale level (reference lib/mask_predictor.py:77)."""
    dev = c2.device
    n_img = c2.shape[0]
    hid = dec.conv1_4.weight.shape[0]
    if (c1 is None) != bool(getattr(dec, "lazy_pred", False)):
        raise K.LavtError("decoder: the 1/4-scale map is omitted exactly when the decoder was built with --lazy_pred")
    y = c4
    levels = []
    plan = [(c3, ("conv1_4", "bn1_4", "conv2_4", "bn2_4")), (c2, ("conv1_3", "bn1_3", "conv2_3", "bn2_3"))]
    if c1 is not None:
        plan.append((c1, ("conv1_2", "bn1_2", "conv2_2", "bn2_2")))
    for skip, (ca, ba, cb, bb) in plan:
        _, H, W, Cs = skip.shape
        if y.shape[1] > H or y.shape[2] > W:
            raise K.LavtError("decoder: coarser map is larger than the skip connection")
        cat = torch.empty(n_img, H, W, y.shape[-1] + Cs, device=dev, dtype=torch.bfloat16)
        K.upsample_concat(y, skip, cat)
        t1, s1 = _cbr_fwd(cat, dec, ca, ba, ws, sync_bn)
        t2, s2 = _cbr_fwd(t1, dec, cb, bb, ws, sync_bn)
        levels.append((tuple(y.shape), s1, s2))
        y = t2
        _count(1)
    # --interpolate_before_seg / --seg_last (reference lib/mask_predictor.py:40-48, 88-97): bilinear x2 + conv3x3 + BN + ReLU at 1/2 scale,
    # and once more at full scale, before the 1x1 classifier
    tails = []
    if getattr(dec, "interpolate_before_seg", False):
        fine = c1
        for on, (cname, bname, mul_) in ((True, ("conv2_1", "bn1_1", 2)), (getattr(dec, "seg_last", False), ("conv1_0", "bn1_0", 4))):
            if not on:
                continue
            up = torch.empty(n_img, mul_ * fine.shape[1], mul_ * fine.shape[2], hid, device=dev, dtype=torch.bfloat16)
            K.upsample_nhwc(y, up)
            t, sv = _cbr_fwd(up, dec, cname, bname, ws, sync_bn)
            tails.append((tuple(y.shape), sv))
            y = t
            _count(1)
    _, H, W, _ = y.shape
    w11 = dec.prepared.get("w11", [dec.conv1_1.weight], lambda: _f32(dec.conv1_1.weight.reshape(2, -1)))
    lg = torch.empty(n_img, H, W, 2, device=dev, dtype=torch.float32)
    K.conv1x1_logits(y.view(-1, hid), w11, dec.conv1_1.bias.detach(), lg.view(-1, 2))
    _count(1)
    return lg, (levels, y, w11, tails)


def decoder_bwd(dec, saved, dlg: torch.Tensor, grads: GradStore, ws: Workspace, sync_bn: bool = False):
    """dlg fp32 [n, H1, W1, 2] -> gradients of (c4, c3, c2, c1) as bf16 row views [n*H_i*W_i, C_i] (c3..c1 are column slices of the
    concatenated-input gradient, i.e. have a row pitch larger than C_i); dc1 is None under --lazy_pred."""
    levels, y, w11, tails = saved
    dev = dlg.device
    hid = y.shape[-1]
    npix = y.shape[0] * y.shape[1] * y.shape[2]
    dy = ws.get("bw_dec_dy", (npix, hid), torch.bfloat16, dev)
    K.conv1x1_logits_bwd(dlg.view(-1, 2), y.view(-1, hid), w11, dy, grads.of(dec.conv1_1.weight).view(2, hid), grads.of(dec.conv1_1.bias))
    _count(1)
    for yshape, sv in reversed(tails):          # adjoint of (bilinear upsample -> conv3x3 + BN + ReLU), finest level first
        up = sv[0]
        dup = torch.empty(up.shape, device=dev, dtype=torch.bfloat16)
        _cbr_bwd(dec, sv, dy, grads, ws, sync_bn, dup)
        dprev = torch.empty(yshape, device=dev, dtype=torch.bfloat16)
        K.upsample_concat_bwd(dup, dprev)
        _count(1)
        dy = dprev.view(-1, hid)
    dskips = []
    for li in range(len(levels) - 1, -1, -1):
        yshape, s1, s2 = levels[li]
        cat = s1[0]
        n, H, W, Ct = cat.shape
        dt1 = ws.get("bw_dec_dt1", (n * H * W, hid), torch.bfloat16, dev)
        _cbr_bwd(dec, s2, dy, grads, ws, sync_bn, dt1.view(n, H, W, hid))
        dcat = torch.empty(n, H, W, Ct, device=dev, dtype=torch.bfloat16)
        _cbr_bwd(dec, s1, dt1, grads, ws, sync_bn, dcat)
        C1 = yshape[-1]
        dskips.append(dcat.view(n * H * W, Ct)[:, C1:])
        dprev = torch.empty(yshape, device=dev, dtype=torch.bfloat16)
        K.upsample_concat_bwd(dcat, dprev)
        _count(1)
        dy = dprev.view(-1, C1)
    dskips = dskips[::-1]                               # coarse -> fine: dc3, dc2(, dc1)
    return (dy, dskips[0], dskips[1], dskips[2] if len(dskips) > 2 else None)       # dc4, dc3, dc2, dc1


# ------------------------------------------------------------------------------------------------
# SepTPWAM + LanguageGate under the README video flags (reference SepTPWAM.forward :1480-1584): every PWAM projection is the sum of
# a Conv3d(3,3,3) branch and a Conv3d(1,1,1) branch
# ------------------------------------------------------------------------------------------------
def conv3d_bwd(dy: torch.Tensor, x5: torch.Tensor, conv, grads: GradStore, ws: Workspace, prepared: E.PreparedWeights, key: str, *,
               dx_bf16: Optional[torch.Tensor] = None, dx_f32: Optional[torch.Tensor] = None, dx_resid: Optional[torch.Tensor] = None) -> None:
    """Adjoint of y = Conv3d_333(x) + b (stride 1, zero padding 1).  dy bf16 [B*D*H*W, Cout]; x5 bf16 [B,D,H,W,Cin].
    dW: 27 split-K GEMMs over the zero-padded transposed layouts (see ``_cbr_bwd``; frames get a zero frame on either side);
    dx = the same implicit-GEMM convolution with flipped taps and Cin <-> Cout."""
    B, D, H, W, Cin = x5.shape
    Cout = conv.weight.shape[0]
    dev = dy.device
    npos = B * D * H * W
    if conv.weight.requires_grad and Cin % 64 == 0:
        # one launch over 5-D TMA boxes (64 channels x 64 pixels of one frame), taps = box offsets, padding = out-of-bounds fill
        K.conv3d_wgrad(dy.view(B, D, H, W, Cout), x5, grads.conv_taps(conv.weight),
                       lambda nfl: ws.get("bw_splitk", (nfl,), torch.float32, dev), accumulate=True)
        _count(2)
    elif conv.weight.requires_grad:
        Wp = _pad8(W + 2)
        Kp = B * (D + 2) * (H + 2) * Wp
        dz_t = ws.get("bw_dzT", (Cout, Kp), torch.bfloat16, dev)
        dz_t.zero_()
        K.nhwc_pad_transpose(dy.view(B * D, H, W, Cout), dz_t, Wp, 0, frames_per_clip=D)
        x_t = ws.get("bw_cxT", (3, Cin, Kp), torch.bfloat16, dev)
        x_t.zero_()
        for kx in range(3):
            K.nhwc_pad_transpose(x5.view(B * D, H, W, Cin), x_t[kx], Wp, kx - 1, frames_per_clip=D)
        gbuf = grads.conv_taps(conv.weight)
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(Cout, Cin, Kp),), torch.float32, dev)
        for tap in range(27):
            kz, ky, kx = tap // 9, (tap // 3) % 3, tap % 3
            K.gemm_bf16_splitk(dz_t, x_t[kx], gbuf[:, tap * Cin:(tap + 1) * Cin], part, accumulate=True,
                               b_koff=(kz - 1) * (H + 2) * Wp + (ky - 1) * Wp)
        _count(6 + 54)
    if conv.bias is not None and conv.bias.requires_grad:
        K.colsum_accumulate(dy, grads.of(conv.bias))
        _count(1)
    if dx_bf16 is not None or dx_f32 is not None:
        def _wT():
            wgt = conv.weight.detach()      # [Cout, Cin, 3, 3, 3] -> [Cin, flipped tap * Cout + co]
            return wgt.flip(2, 3, 4).permute(1, 2, 3, 4, 0).reshape(wgt.shape[1], -1).to(torch.bfloat16).contiguous()
        w_t = prepared.get(key + "_wT", [conv.weight], _wT)
        K.conv3d_bf16(dy.view(B, D, H, W, Cout), w_t, out_bf16=dx_bf16, out_f32=dx_f32, resid=dx_resid)
        _count(1)


def sep_t_pwam_gate_fwd(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, D: int, H: int,
                        W: int, ws: Workspace, gate_act: str = "tanh"):
    """Training twin of ``engine.sep_t_pwam_gate``: returns (r fp32 [B*n, C], gated x or None, saved)."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    heads = fusion.num_heads
    Nl = l.shape[-1]
    bf, f32 = torch.bfloat16, torch.float32

    def w333(name, conv):
        return pw.get(name, [conv.weight], lambda: _bf16(conv.weight.detach().permute(0, 2, 3, 4, 1).reshape(conv.weight.shape[0], -1)))

    def w111(name, conv):
        return pw.get(name, [conv.weight], lambda: _bf16(conv.weight.detach().reshape(conv.weight.shape[0], -1)))

    def b_(conv):
        return conv.bias.detach()

    def rows(dtype):
        return torch.empty(N_, C, device=dev, dtype=dtype)
    xb5 = xb.view(B, D, H, W, C)
    t32 = ws.get("sp_t32", (N_, C), f32, dev)
    scr32 = ws.get("sp_scr32", (N_, C), f32, dev)
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(B, n, C),), f32, dev)
    ident = pw.get("ident_%d_%s" % (B, dev), [], lambda: torch.stack([torch.zeros(B, C), torch.ones(B, C)], 1).to(dev).contiguous())
    # ts_vis = GELU(conv333(x)) + GELU(conv111(x))
    vt, vs_ = fusion.temporal_vis_project[0], fusion.spatial_vis_project[0]
    vt_pre, vs_pre, vis = rows(bf), rows(bf), rows(bf)
    K.conv3d_bf16(xb5, w333("vis_t", vt), bias=b_(vt), out_bf16=vt_pre)
    K.gemm_bf16(xb, w111("vis_s", vs_), bias=b_(vs_), out_bf16=vs_pre)
    K.gate_elementwise(3, vt_pre, out_bf16=vis, out_f32=t32)
    K.gate_elementwise(5, vs_pre, f=t32, out_bf16=vis, out_f32=scr32)
    # query = IN3d(conv333(x)) + IN3d(conv111(x))
    qt, qs_ = fusion.f_query_t[0], fusion.f_query_s[0]
    qa, qb, qhat = (torch.empty(B, n, C, device=dev, dtype=f32) for _ in range(3))
    sa_q, sb_q = (torch.empty(B, 2, C, device=dev, dtype=f32) for _ in range(2))
    K.conv3d_bf16(xb5, w333("q_t", qt), bias=b_(qt), out_f32=qa.view(N_, C))
    K.gemm_bf16(xb, w111("q_s", qs_), bias=b_(qs_), out_f32=qb.view(N_, C))
    K.instnorm_stats(qa, sa_q, stw)
    K.instnorm_stats(qb, sb_q, stw)
    K.instnorm_sum2(qa, sa_q, qb, sb_q, qhat)
    k_w = pw.get("k_w", [fusion.f_key[0].weight], lambda: _f32(fusion.f_key[0].weight[:, :, 0]))
    v_w = pw.get("v_w", [fusion.f_value[0].weight], lambda: _f32(fusion.f_value[0].weight[:, :, 0]))
    kk = torch.empty(B, Nl, C, device=dev, dtype=f32)
    vv = torch.empty(B, Nl, C, device=dev, dtype=f32)
    K.pwam_kv(l, mask, k_w, b_(fusion.f_key[0]), v_w, b_(fusion.f_value[0]), kk, vv)
    o = torch.empty(B, n, C, device=dev, dtype=bf)
    K.pwam_attend(qhat, ident, kk, vv, mask, o, heads)
    # lang = IN3d(conv333(o)) + IN3d(conv111(o))
    Wt, Ws = fusion.W_t[0], fusion.W_s[0]
    la, lb, lang = (torch.empty(B, n, C, device=dev, dtype=f32) for _ in range(3))
    sa_l, sb_l = (torch.empty(B, 2, C, device=dev, dtype=f32) for _ in range(2))
    K.conv3d_bf16(o.view(B, D, H, W, C), w333("W_t", Wt), bias=b_(Wt), out_f32=la.view(N_, C))
    K.gemm_bf16(o.view(N_, C), w111("W_s", Ws), bias=b_(Ws), out_f32=lb.view(N_, C))
    K.instnorm_stats(la, sa_l, stw)
    K.instnorm_stats(lb, sb_l, stw)
    K.instnorm_sum2(la, sa_l, lb, sb_l, lang)
    a2 = torch.empty(B, n, C, device=dev, dtype=bf)
    K.pwam_mul_norm(vis.view(B, n, C), lang, ident, a2)
    # r = GELU(conv333(mm)) + GELU(conv111(mm))
    mt, ms = fusion.project_mm_t[0], fusion.project_mm_s[0]
    rt_pre, rs_pre, rb = rows(bf), rows(bf), rows(bf)
    r32 = rows(f32)
    K.conv3d_bf16(a2.view(B, D, H, W, C), w333("mm_t", mt), bias=b_(mt), out_bf16=rt_pre)
    K.gemm_bf16(a2.view(N_, C), w111("mm_s", ms), bias=b_(ms), out_bf16=rs_pre)
    K.gate_elementwise(3, rt_pre, out_bf16=rb, out_f32=t32)
    K.gate_elementwise(5, rs_pre, f=t32, out_bf16=rb, out_f32=r32)
    _count(27)
    g1 = g2 = xg = None
    if res_gate is not None:
        g0w = pw.get("g0", [res_gate[0].weight], lambda: _bf16(res_gate[0].weight))
        g2w = pw.get("g2", [res_gate[2].weight], lambda: _bf16(res_gate[2].weight))
        g1, g2 = rows(bf), rows(bf)
        K.gemm_bf16(rb, g0w, act=K.ACT_RELU, out_bf16=g1)
        K.gemm_bf16(g1, g2w, out_bf16=g2)
        xg = rows(f32)
        K.gate_elementwise(0 if gate_act == "tanh" else 7, g2, rb, f=x, out_f32=xg)      # --lg_act_layer sigmoid: modes 7 / 8
        _count(3)
    saved = dict(xb=xb, vt_pre=vt_pre, vs_pre=vs_pre, vis=vis, qa=qa, qb=qb, qhat=qhat, sa_q=sa_q, sb_q=sb_q, kk=kk, vv=vv, o=o, la=la,
                 lb=lb, lang=lang, sa_l=sa_l, sb_l=sb_l, a2=a2, rt_pre=rt_pre, rs_pre=rs_pre, rb=rb, g1=g1, g2=g2, l=l, mask=mask, B=B,
                 dims=(D, H, W), heads=heads, k_w=k_w, v_w=v_w, ident=ident, gate_act=gate_act)
    return r32, xg, saved


def sep_t_pwam_gate_bwd(fusion, res_gate, saved, dr_out: Optional[torch.Tensor], dxg: Optional[torch.Tensor], grads: GradStore,
                        ws: Workspace, dl: torch.Tensor) -> torch.Tensor:
    """Adjoint of ``sep_t_pwam_gate_fwd`` (same contract as ``pwam_gate_bwd``)."""
    s = saved
    B, heads = s["B"], s["heads"]
    D, H, W = s["dims"]
    xb = s["xb"]
    N_, C = xb.shape
    n = N_ // B
    dev = xb.device
    bf, f32 = torch.bfloat16, torch.float32
    pw = fusion.prepared
    ident = s["ident"]
    Nl = s["l"].shape[-1]
    nlp = _nl_pad(Nl)

    def wsb(name, dtype=bf):
        return ws.get("bw_sp_" + name, (N_, C), dtype, dev)
    dr = dr_out
    if res_gate is not None and dxg is not None:
        dg2pre = wsb("a")
        gmode = 1 if s.get("gate_act", "tanh") == "tanh" else 8
        if dr is None:
            dr = wsb("dr", f32)
            K.gate_elementwise(gmode, s["g2"], s["rb"], f=dxg, f2=None, out_bf16=dg2pre, out_f32=dr)
        else:
            K.gate_elementwise(gmode, s["g2"], s["rb"], f=dxg, f2=dr, out_bf16=dg2pre, out_f32=dr)
        dg1 = wsb("b")
        linear_bwd(dg2pre, s["g1"], res_gate[2].weight, None, grads, ws, pw, "g2", dx_bf16=dg1)
        K.gate_elementwise(2, dg1, s["g1"], out_bf16=dg1)
        linear_bwd(dg1, s["rb"], res_gate[0].weight, None, grads, ws, pw, "g0", dx_f32=dr, dx_resid=dr)
        _count(2)
    if dr is None:
        raise K.LavtError("SepTPWAM backward: neither the stage output nor the gated features carry a gradient")
    a2 = s["a2"].view(N_, C)
    o = s["o"].view(N_, C)
    vis = s["vis"]
    # r = GELU(rt_pre) + GELU(rs_pre)
    drt, drs = wsb("a"), wsb("b")
    K.gate_elementwise(4, s["rt_pre"], f=dr, out_bf16=drt)
    K.gate_elementwise(4, s["rs_pre"], f=dr, out_bf16=drs)
    acc32 = wsb("acc32", f32)
    da2 = wsb("c")
    mt, ms = fusion.project_mm_t[0], fusion.project_mm_s[0]
    linear_bwd(drs, a2, ms.weight, ms.bias, grads, ws, pw, "mm_s", dx_f32=acc32)
    conv3d_bwd(drt, a2.view(B, D, H, W, C), mt, grads, ws, pw, "mm_t", dx_bf16=da2, dx_resid=acc32)
    # a2 = vis * (IN(la) + IN(lb)),  vis = GELU(vt_pre) + GELU(vs_pre)
    sums = torch.zeros(6, B, 2, C, device=dev, dtype=f32)
    scratch, dvt, dvs = wsb("a"), wsb("d"), wsb("e")
    K.pwam_mul_norm_bwd(da2, vis, s["vt_pre"], s["la"], s["sa_l"], scratch, sums[0])        # reductions of the temporal branch
    K.pwam_mul_norm_bwd(da2, vis, s["vt_pre"], s["lb"], s["sb_l"], scratch, sums[1])        # ... of the spatial branch
    K.pwam_mul_norm_bwd(da2, vis, s["vt_pre"], s["lang"], ident, dvt, sums[2])              # d vt_pre = da2 * lang * GELU'(vt_pre)
    K.pwam_mul_norm_bwd(da2, vis, s["vs_pre"], s["lang"], ident, dvs, sums[3])
    dla, dlb = wsb("a"), wsb("b")
    K.instnorm_bwd(s["la"], s["sa_l"], sums[0], dla, ga=da2, gb=vis)
    K.instnorm_bwd(s["lb"], s["sb_l"], sums[1], dlb, ga=da2, gb=vis)
    Wt, Ws = fusion.W_t[0], fusion.W_s[0]
    do = wsb("c")
    linear_bwd(dlb, o, Ws.weight, Ws.bias, grads, ws, pw, "W_s", dx_f32=acc32)
    conv3d_bwd(dla, o.view(B, D, H, W, C), Wt, grads, ws, pw, "W_t", dx_bf16=do, dx_resid=acc32)
    # pixel-word attention core on q^ = IN(qa) + IN(qb)
    Wd = B * heads * nlp
    dqhat = ws.get("bw_pw_dq", (B, n, C), f32, dev)
    qs = wsb("a")
    p_bd = ws.get("bw_pw_pbd", (N_, Wd), bf, dev)
    ds_bd = ws.get("bw_pw_dsbd", (N_, Wd), bf, dev)
    K.pwam_attend_bwd(s["qhat"], ident, s["kk"], s["vv"], s["mask"], do, dqhat, qs, p_bd, ds_bd, sums[2], heads, nlp)
    dkv = torch.empty(2, Wd, C, device=dev, dtype=f32)
    for buf, dy_rows, x_rows in ((dkv[0], ds_bd, qs), (dkv[1], p_bd, do)):
        part = ws.get("bw_splitk", (K.splitk_workspace_floats(Wd, C, N_),), f32, dev)
        K.gemm_bf16_wgrad(dy_rows, x_rows, buf, part, accumulate=False)
    fk, fv = fusion.f_key[0], fusion.f_value[0]
    K.pwam_kv_bwd(dkv[0], dkv[1], s["mask"], s["l"], s["k_w"], s["v_w"],
                  grads.of(fk.weight) if fk.weight.requires_grad else None, grads.of(fk.bias) if fk.bias.requires_grad else None,
                  grads.of(fv.weight) if fv.weight.requires_grad else None, grads.of(fv.bias) if fv.bias.requires_grad else None,
                  dl, heads, nlp)
    K.instnorm_bwd_reduce(dqhat, s["qa"], s["sa_q"], sums[4])
    K.instnorm_bwd_reduce(dqhat, s["qb"], s["sb_q"], sums[5])
    dqa, dqb = wsb("b"), wsb("c")
    K.instnorm_bwd(s["qa"], s["sa_q"], sums[4], dqa, g_f32=dqhat)
    K.instnorm_bwd(s["qb"], s["sb_q"], sums[5], dqb, g_f32=dqhat)
    # the four projections of x
    if dxg is not None:
        dx, first = dxg, dxg
    else:
        dx, first = torch.empty(N_, C, device=dev, dtype=f32), None
    vt, vs_ = fusion.temporal_vis_project[0], fusion.spatial_vis_project[0]
    qt, qs_ = fusion.f_query_t[0], fusion.f_query_s[0]
    xb5 = xb.view(B, D, H, W, C)
    linear_bwd(dvs, xb, vs_.weight, vs_.bias, grads, ws, pw, "vis_s", dx_f32=dx, dx_resid=first)
    linear_bwd(dqb, xb, qs_.weight, qs_.bias, grads, ws, pw, "q_s", dx_f32=dx, dx_resid=dx)
    conv3d_bwd(dvt, xb5, vt, grads, ws, pw, "vis_t", dx_f32=dx, dx_resid=dx)
    conv3d_bwd(dqa, xb5, qt, grads, ws, pw, "q_t", dx_f32=dx, dx_resid=dx)
    _count(24)
    return dx
