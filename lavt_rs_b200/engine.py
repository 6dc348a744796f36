"""Host-side execution engine: sequences the sm_100a kernels for each reference function.

Layout in HBM
  * residual stream  x : fp32 [B*D*H*W, C] channels-last (the reference's (B,D,H,W,C) view)
  * GEMM operands      : bf16 rows (tokens x C), produced by the LN / gather / epilogue kernels
  * weights            : bf16 [out, in] copies of the fp32 parameters (``PreparedWeights``), refreshed
                         whenever a parameter's version counter changes
Scratch buffers come from a per-device ``Workspace`` so that a steady-state forward performs no
allocations (required for CUDA-graph capture in bench.py).

No reference code path is used here; each function cites the reference function it replaces.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _cabi as K
from .geometry import window_geometry

LAUNCHES = 0  # number of our kernel launches issued (bench.py reports it)
PRECISION = "bf16"   # "fp32": the Swin block runs on the fp32 validation twins (csrc/fp32_ref_kernels.cu); see set_precision


def set_precision(mode: str) -> str:
    """'bf16' (production: bf16 operands on tcgen05, fp32 accumulation) or 'fp32' (validation: fp32 operands and activations through
    the whole Swin block on the CUDA-core twins -- north_star's "1e-4 in fp32 with fp32 accumulate" mode).  Returns the previous mode."""
    global PRECISION
    if mode not in ("bf16", "fp32"):
        raise ValueError("precision must be 'bf16' or 'fp32'")
    prev, PRECISION = PRECISION, mode
    return prev


def _count(n: int = 1) -> None:
    global LAUNCHES
    LAUNCHES += n


class Workspace:
    """Named scratch buffers, grown on demand and reused across calls (one per device / stream user)."""

    def __init__(self):
        self._bufs: Dict[Tuple[str, torch.dtype], torch.Tensor] = {}

    def get(self, name: str, shape: Sequence[int], dtype: torch.dtype, device) -> torch.Tensor:
        numel = 1
        for s in shape:
            numel *= int(s)
        key = (name, dtype)
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < numel or buf.device != torch.device(device):
            buf = torch.empty(max(numel, 1), dtype=dtype, device=device)
            self._bufs[key] = buf
        return buf[:numel].view(*shape)

    def bytes(self) -> int:
        return sum(b.numel() * b.element_size() for b in self._bufs.values())


_WORKSPACES: Dict[Tuple[int, str], Workspace] = {}


def workspace(device, tag: str = "main") -> Workspace:
    dev = torch.device(device)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), tag)
    if key not in _WORKSPACES:
        _WORKSPACES[key] = Workspace()
    return _WORKSPACES[key]


class PreparedWeights:
    """bf16 / folded copies of a module's parameters, rebuilt when any source tensor changes."""

    def __init__(self):
        self._cache: Dict[str, Tuple[tuple, object]] = {}

    def get(self, key: str, sources: Sequence[torch.Tensor], build):
        ver = tuple((t.data_ptr(), t._version, t.device) for t in sources)
        hit = self._cache.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        with torch.no_grad():
            val = build()
        self._cache[key] = (ver, val)
        return val

    def clear(self):
        self._cache.clear()


def _bf16(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.bfloat16).contiguous()


def _f32(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise K.LavtError(f"{what} must live on a CUDA device: the B200 path has no CPU fallback")


# ------------------------------------------------------------------------------------------------
# Swin block  (reference SwinTransformerBlock3D.forward, lib/video_swin_transformer.py:253-273)
# ------------------------------------------------------------------------------------------------
def swin_block(x: torch.Tensor, blk, B: int, D: int, H: int, W: int, window, shifted: bool, clamp: bool,
               ws: Workspace, xb_out: Optional[torch.Tensor] = None) -> None:
    """In place on the fp32 residual stream x [B*D*H*W, C].  ``blk`` is a host SwinTransformerBlock3D.
    If ``xb_out`` is given the final value of x is also written there in bf16 (feeds PWAM's GEMMs)."""
    n, C = x.shape
    dev = x.device
    geom = window_geometry(B, D, H, W, window, shifted, clamp)
    rows = geom.rows()
    nH = blk.num_heads
    pw = blk.prepared
    hd = C // nH
    if PRECISION == "fp32":
        return _swin_block_fp32(x, blk, geom, ws, xb_out)

    qkv_w = pw.get("qkv_w", [blk.attn.qkv.weight], lambda: _bf16(blk.attn.qkv.weight))
    # q columns are scaled by head_dim^-0.5 (:147) times log2(e) in the epilogue -- the attention kernel's softmax
    # runs in base 2:  (acc + b) * s == acc * s + b * s
    def _qscale():
        s = torch.ones(3 * C, device=dev, dtype=torch.float32)
        s[:C] = hd ** -0.5 * 1.4426950408889634
        b = _f32(blk.attn.qkv.bias) * s if blk.attn.qkv.bias is not None else torch.zeros(3 * C, device=dev)
        return s, b
    qkv_s, qkv_b = pw.get("qkv_sb", [blk.attn.qkv.weight] + ([blk.attn.qkv.bias] if blk.attn.qkv.bias is not None else []), _qscale)
    proj_w = pw.get("proj_w", [blk.attn.proj.weight], lambda: _bf16(blk.attn.proj.weight))
    fc1_w = pw.get("fc1_w", [blk.mlp.fc1.weight], lambda: _bf16(blk.mlp.fc1.weight))
    fc2_w = pw.get("fc2_w", [blk.mlp.fc2.weight], lambda: _bf16(blk.mlp.fc2.weight))
    table_t = pw.get("table_t", [blk.attn.relative_position_bias_table],
                     lambda: _f32(blk.attn.relative_position_bias_table.t()))

    # --- attention half: LN1 + shift + partition gather -> qkv GEMM -> window attention -> proj GEMM + scatter + residual
    xw = ws.get("xw", (rows, C), torch.bfloat16, dev)
    K.layernorm_window_gather(x, geom, blk.norm1.weight, blk.norm1.bias, xw, eps=blk.norm1.eps)
    qkv = ws.get("qkv", (rows, 3 * C), torch.bfloat16, dev)
    K.gemm_bf16(xw, qkv_w, cscale=qkv_s, bias=qkv_b, out_bf16=qkv)
    att = ws.get("att", (rows, C), torch.bfloat16, dev)
    K.window_attention(qkv, table_t, geom, att)
    K.gemm_bf16(att, proj_w, bias=blk.attn.proj.bias.detach(), resid=x, out_f32=x, win=geom)
    # --- MLP half: LN2 -> fc1 + GELU -> fc2 + residual
    h1 = ws.get("ln2", (n, C), torch.bfloat16, dev)
    K.layernorm_rows(x, blk.norm2.weight, blk.norm2.bias, out_bf16=h1, eps=blk.norm2.eps)
    hid = ws.get("hid", (n, fc1_w.shape[0]), torch.bfloat16, dev)
    K.gemm_bf16(h1, fc1_w, bias=blk.mlp.fc1.bias.detach(), act=K.ACT_GELU, out_bf16=hid)
    K.gemm_bf16(hid, fc2_w, bias=blk.mlp.fc2.bias.detach(), resid=x, out_f32=x, out_bf16=xb_out)
    _count(7)


def _swin_block_fp32(x: torch.Tensor, blk, geom, ws: Workspace, xb_out: Optional[torch.Tensor]) -> None:
    """Same launch sequence as ``swin_block`` with fp32 operands / activations on the validation twins (no bf16 rounding anywhere)."""
    n, C = x.shape
    dev = x.device
    rows, nH = geom.rows(), blk.num_heads
    hd = C // nH
    s = torch.ones(3 * C, device=dev, dtype=torch.float32)
    s[:C] = hd ** -0.5 * 1.4426950408889634
    qb = _f32(blk.attn.qkv.bias) * s if blk.attn.qkv.bias is not None else torch.zeros(3 * C, device=dev)
    xw = ws.get("xw32", (rows, C), torch.float32, dev)
    K.layernorm_window_gather_f32(x, geom, blk.norm1.weight, blk.norm1.bias, xw, eps=blk.norm1.eps)
    qkv = ws.get("qkv32", (rows, 3 * C), torch.float32, dev)
    K.gemm_f32_ref(xw, _f32(blk.attn.qkv.weight), cscale=s, bias=qb, out_f32=qkv)
    att = ws.get("att32", (rows, C), torch.float32, dev)
    K.window_attention_f32_ref(qkv, _f32(blk.attn.relative_position_bias_table.t()), geom, att)
    K.gemm_f32_ref(att, _f32(blk.attn.proj.weight), bias=blk.attn.proj.bias.detach(), resid=x, out_f32=x, win=geom)
    h1 = ws.get("ln2_32", (n, C), torch.float32, dev)
    K.layernorm_rows(x, blk.norm2.weight, blk.norm2.bias, out_f32=h1, eps=blk.norm2.eps)
    hid = ws.get("hid32", (n, blk.mlp.fc1.weight.shape[0]), torch.float32, dev)
    K.gemm_f32_ref(h1, _f32(blk.mlp.fc1.weight), bias=blk.mlp.fc1.bias.detach(), act=K.ACT_GELU, out_f32=hid)
    K.gemm_f32_ref(hid, _f32(blk.mlp.fc2.weight), bias=blk.mlp.fc2.bias.detach(), resid=x, out_f32=x, out_bf16=xb_out)
    _count(7)


# ------------------------------------------------------------------------------------------------
# PWAM + LanguageGate  (reference PWAM.forward :919-934, SpatialImageLanguageAttention.forward :975-1009,
# res_gate :519-525 applied at :570)
# ------------------------------------------------------------------------------------------------
def _conv1x1_w(conv) -> torch.Tensor:
    return conv.weight[:, :, 0]


def _language_gate(x: torch.Tensor, rb: torch.Tensor, res_gate, pw: PreparedWeights, scratch: torch.Tensor, gate_act: str) -> None:
    """LanguageGate (reference res_gate :519-525 applied at :570; 2-D lib/backbone.py:599-609): x += act(W2 relu(W1 r)) * r as two GEMMs
    whose epilogues carry ReLU and tanh | sigmoid (--lg_act_layer), the elementwise product and the residual add.  ``scratch`` is a dead
    bf16 [n, C] buffer of the caller."""
    if res_gate is None:
        return
    if gate_act not in ("tanh", "sigmoid"):
        raise K.LavtError(f"LanguageGate activation {gate_act!r}: the reference offers tanh and sigmoid (--lg_act_layer)")
    g0 = pw.get("g0", [res_gate[0].weight], lambda: _bf16(res_gate[0].weight))
    g2 = pw.get("g2", [res_gate[2].weight], lambda: _bf16(res_gate[2].weight))
    K.gemm_bf16(rb, g0, act=K.ACT_RELU, out_bf16=scratch)
    K.gemm_bf16(scratch, g2, act=K.ACT_TANH if gate_act == "tanh" else K.ACT_SIGMOID, mul=rb, resid=x, out_f32=x)
    _count(2)


def pwam_gate(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int,
              ws: Workspace, gate_act: str = "tanh", r_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x fp32 [B*n, C] (updated in place with the gated residual), xb = bf16 copy of x, l fp32 [B,768,Nl],
    mask fp32 [B,Nl].  Returns r (= x_residual) as fp32 [B*n, C]."""
    if getattr(fusion, "kind", "pwam") == "gacd":
        return gacd_gate(x, xb, fusion, res_gate, l, mask, B, ws, gate_act=gate_act, r_f32=r_f32)
    if getattr(fusion, "kind", "pwam") == "bcam":
        return bcam_gate(x, xb, fusion, res_gate, l, mask, B, ws, gate_act=gate_act, r_f32=r_f32)
    if getattr(fusion, "kind", "pwam") == "efn":
        return efn_gate(x, xb, fusion, res_gate, l, mask, B, ws, gate_act=gate_act, r_f32=r_f32)
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    att = fusion.image_lang_att
    Nl = l.shape[-1]

    def wprep(name, conv):
        return pw.get(name, [conv.weight], lambda: _bf16(_conv1x1_w(conv)))

    if not fusion.attention:
        # --fuse simple (reference :916-917, :929-930): lang = LangProject(mean-pooled words), one vector per clip
        vis = ws.get("pw_vis", (B, n, C), torch.bfloat16, dev)
        K.gemm_bf16(xb, wprep("vis_w", fusion.vis_project[0]), bias=fusion.vis_project[0].bias.detach(), act=K.ACT_GELU, out_bf16=vis.view(N_, C))
        stats = ws.get("pw_stats", (B, 2, C), torch.float32, dev)
        pr = att.project
        K.lang_project(l, mask, _f32(pr[0].weight), _f32(pr[0].bias), _f32(pr[2].weight), _f32(pr[2].bias), stats)
        zeros = pw.get("zeros_%d_%d" % (B, n), [], lambda: torch.zeros(B, n, C, device=dev, dtype=torch.float32))
        a2 = ws.get("pw_o", (B, n, C), torch.bfloat16, dev)
        K.pwam_mul_norm(vis, zeros, stats, a2)          # vis * (0 - (-lang)) * 1
        r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
        rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
        K.gemm_bf16(a2.view(N_, C), wprep("mm_w", fusion.project_mm[0]), bias=fusion.project_mm[0].bias.detach(), act=K.ACT_GELU, out_f32=r32,
                    out_bf16=rb)
        _count(6)
        _language_gate(x, rb, res_gate, pw, vis.view(N_, C), gate_act)
        return r32
    heads = att.num_heads

    vis_w = wprep("vis_w", fusion.vis_project[0])
    q_w = wprep("q_w", att.f_query[0])
    W_w = wprep("W_w", att.W[0])
    mm_w = wprep("mm_w", fusion.project_mm[0])
    k_w = pw.get("k_w", [att.f_key[0].weight], lambda: _f32(_conv1x1_w(att.f_key[0])))
    v_w = pw.get("v_w", [att.f_value[0].weight], lambda: _f32(_conv1x1_w(att.f_value[0])))

    vis = ws.get("pw_vis", (B, n, C), torch.bfloat16, dev)
    K.gemm_bf16(xb, vis_w, bias=fusion.vis_project[0].bias.detach(), act=K.ACT_GELU, out_bf16=vis.view(N_, C))
    qpre = ws.get("pw_q", (B, n, C), torch.float32, dev)      # fp32: feeds InstanceNorm + SIMT attention, never an MMA operand
    stats = ws.get("pw_stats", (B, 2, C), torch.float32, dev)
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(B, n, C),), torch.float32, dev)
    # --att_norm_layer_type (2-D backbone, reference lib/backbone.py:1297-1316): IN = per-image statistics over the tokens (default);
    # BN (eval) folds into the producing GEMM's column scale / bias; LN is a row LayerNorm of the GEMM result; none = identity.
    # For the last three the consumers read "statistics" (mean 0, rstd 1).
    norm_kind = getattr(att, "att_norm_layer_type", "IN")
    ident = None
    if norm_kind != "IN":
        ident = pw.get("ident_%d_%s" % (B, dev), [], lambda: torch.stack([torch.zeros(B, C), torch.ones(B, C)], 1).to(dev).contiguous())

    def normed_gemm(a_rows, w, seq, tag, out32):
        """out32 = norm(conv1x1(a_rows)) for BN / LN / none; for IN the plain projection (statistics computed by the caller)."""
        bias = seq[0].bias.detach()
        if norm_kind == "BN":
            bn = seq[1]
            if bn.training:
                raise K.LavtError("--att_norm_layer_type BN is inference-only on the B200 path (BatchNorm must be in eval mode)")
            sc, sh = pw.get(tag + "_bn", [bn.weight, bn.bias, bn.running_mean, bn.running_var, seq[0].bias],
                            lambda: (lambda s_, t_: (s_, (_f32(seq[0].bias) * s_ + t_).contiguous()))(*_bn_fold(bn)))
            K.gemm_bf16(a_rows, w, cscale=sc, bias=sh, out_f32=out32)
        else:
            K.gemm_bf16(a_rows, w, bias=bias, out_f32=out32)
            if norm_kind == "LN":
                K.layernorm_rows(out32, seq[1].weight, seq[1].bias, out_f32=out32, eps=seq[1].eps)
                _count(1)
    normed_gemm(xb, q_w, att.f_query, "fq", qpre.view(N_, C))
    if norm_kind == "IN":
        K.instnorm_stats(qpre, stats, stw)
    kk = ws.get("pw_k", (B, Nl, C), torch.float32, dev)
    vv = ws.get("pw_v", (B, Nl, C), torch.float32, dev)
    K.pwam_kv(l, mask, k_w, att.f_key[0].bias.detach(), v_w, att.f_value[0].bias.detach(), kk, vv)
    o = ws.get("pw_o", (B, n, C), torch.bfloat16, dev)
    K.pwam_attend(qpre, stats if norm_kind == "IN" else ident, kk, vv, mask, o, heads)
    lang = qpre  # q_pre is dead: reuse its buffer for lang_pre
    normed_gemm(o.view(N_, C), W_w, att.W, "W", lang.view(N_, C))
    if norm_kind == "IN":
        K.instnorm_stats(lang, stats, stw)
    a2 = o  # o is dead after the W projection
    K.pwam_mul_norm(vis, lang, stats if norm_kind == "IN" else ident, a2)
    r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
    rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
    K.gemm_bf16(a2.view(N_, C), mm_w, bias=fusion.project_mm[0].bias.detach(), act=K.ACT_GELU, out_f32=r32, out_bf16=rb)
    _count(11)
    _language_gate(x, rb, res_gate, pw, vis.view(N_, C), gate_act)      # vis is dead: scratch
    return r32


def gacd_gate(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, ws: Workspace,
              gate_act: str = "tanh", r_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """GA-CD fusion (reference lib/bcam.py:78-127, --gacd) + LanguageGate; same contract as ``pwam_gate``."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    stats = ws.get("pw_stats", (B, 2, C), torch.float32, dev)
    pr = fusion.lang_gen.project
    K.lang_project(l, mask, _f32(pr[0].weight), _f32(pr[0].bias), _f32(pr[2].weight), _f32(pr[2].bias), stats)      # (-ls, 1)
    zeros = pw.get("zeros_%d_%d" % (B, n), [], lambda: torch.zeros(B, n, C, device=dev, dtype=torch.float32))
    a = ws.get("pw_o", (B, n, C), torch.bfloat16, dev)
    K.pwam_mul_norm(xb.view(B, n, C), zeros, stats, a)                                        # ls * x
    xm = ws.get("pw_q", (B, n, C), torch.float32, dev)
    mm = fusion.mm_gen[0]
    K.gemm_bf16(a.view(N_, C), pw.get("mm_w", [mm.weight], lambda: _bf16(mm.weight)), bias=mm.bias.detach(), act=K.ACT_RELU,
                out_f32=xm.view(N_, C))
    r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
    rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
    K.gacd_fuse(xm, stats, _f32(fusion.query.weight), _f32(fusion.query.bias), _f32(fusion.key_c.weight), _f32(fusion.key_c.bias),
                _f32(fusion.key_d.weight), _f32(fusion.key_d.bias), _f32(fusion.value.weight), _f32(fusion.value.bias),
                lambda nfl: ws.get("gacd_ws", (nfl,), torch.float32, dev), out_f32=r32, out_bf16=rb)
    _count(10)
    _language_gate(x, rb, res_gate, pw, a.view(N_, C), gate_act)        # the ls * x operand is dead: scratch
    return r32


def bcam_gate(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, ws: Workspace,
              gate_act: str = "tanh", r_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """BCAM fusion (reference lib/bcam.py:43-75, --bcam) + LanguageGate; same contract as ``pwam_gate``.  Eleven tcgen05 GEMMs with
    the three ``csrc/bcam_kernels.cu`` kernels between them; sums of two Linear layers run as one GEMM over row-concatenated operands
    (one [n, 3C] buffer holds out2 | out | query2, so cat[out2, out] and [out | query2] are column windows of it, never copies).
    The hw x hw relation map (:61-62) is materialised once as fp32 logits and once as bf16 probabilities (1.2 GB at 120 x 120)."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    if n != fusion.hw:
        raise K.LavtError(f"BCAM: a_proj maps to {fusion.hw} positions but the feature map has {n} (the reference pins --bcam to 480 x 480 inputs)")
    pw = fusion.prepared
    Nl = l.shape[-1]
    Nlp = (Nl + 31) // 32 * 32           # N granule of the sim GEMM (also a K granule of the out GEMM)
    hwp = (n + 31) // 32 * 32            # N granule of a_proj
    hw8 = (n + 7) // 8 * 8               # K granule of rel_map @ query3

    def wb(name, lin):
        return pw.get(name, [lin.weight], lambda: _bf16(lin.weight))

    def b_(lin):
        return lin.bias.detach()

    lr = ws.get("bc_lr", (B, Nlp, C), torch.bfloat16, dev)
    lrT = ws.get("bc_lrT", (B, C, Nlp), torch.bfloat16, dev)
    K.bcam_words(l, _f32(fusion.lang_reduce.weight), _f32(fusion.lang_reduce.bias), lr, lrT)
    # VLAM (:51-56): sim = softmax(relu(vis_1 x) lr^T + mask), out = sim lr
    q = ws.get("pw_vis", (N_, C), torch.bfloat16, dev)
    K.gemm_bf16(xb, wb("v1_w", fusion.vis_1[0]), bias=b_(fusion.vis_1[0]), act=K.ACT_RELU, out_bf16=q)
    sim = ws.get("bc_sim", (N_, Nlp), torch.float32, dev)
    for b in range(B):
        K.gemm_bf16(q[b * n:(b + 1) * n], lr[b], out_f32=sim[b * n:(b + 1) * n])
    simp = ws.get("bc_simp", (N_, Nlp), torch.bfloat16, dev)
    K.bcam_softmax_rows(sim, Nl, simp, mask=mask, rows_per_mask=n)
    cat = ws.get("bc_cat", (N_, 3 * C), torch.bfloat16, dev)        # out2 | out | query2
    for b in range(B):
        K.gemm_bf16(simp[b * n:(b + 1) * n], lrT[b], out_bf16=cat[b * n:(b + 1) * n, C:2 * C])
    # LVAM (:59-64): A = tanh(out_1(out) + vis_2_2(relu(vis_2 x))); rel_map = softmax(a_proj(A)); out2 = rel_map relu(vis_3 x)
    K.gemm_bf16(xb, wb("v2_w", fusion.vis_2[0]), bias=b_(fusion.vis_2[0]), act=K.ACT_RELU, out_bf16=cat[:, 2 * C:])
    w_a = pw.get("a_w", [fusion.out_1.weight, fusion.vis_2_2.weight], lambda: _bf16(torch.cat([fusion.out_1.weight, fusion.vis_2_2.weight], 1)))
    b_a = pw.get("a_b", [fusion.out_1.bias, fusion.vis_2_2.bias], lambda: _f32(fusion.out_1.bias + fusion.vis_2_2.bias))
    a = ws.get("pw_o", (N_, C), torch.bfloat16, dev)
    K.gemm_bf16(cat[:, C:], w_a, bias=b_a, act=K.ACT_TANH, out_bf16=a)

    def _aproj():
        w = torch.zeros(hwp, C, device=dev, dtype=torch.bfloat16)
        w[:n] = fusion.a_proj.weight.detach()
        bb = torch.zeros(hwp, device=dev, dtype=torch.float32)
        bb[:n] = fusion.a_proj.bias.detach()
        return w, bb
    ap_w, ap_b = pw.get("ap", [fusion.a_proj.weight, fusion.a_proj.bias], _aproj)
    logits = ws.get("bc_logits", (N_, hwp), torch.float32, dev)
    K.gemm_bf16(a, ap_w, bias=ap_b, out_f32=logits)
    rel = ws.get("bc_rel", (N_, hwp), torch.bfloat16, dev)
    K.bcam_softmax_rows(logits, n, rel)
    K.gemm_bf16(xb, wb("v3_w", fusion.vis_3[0]), bias=b_(fusion.vis_3[0]), act=K.ACT_RELU, out_bf16=q)         # query is dead: query3
    q3T = ws.get("bc_q3T", (B, C, hw8), torch.bfloat16, dev)
    K.bcam_transpose_pad(q, q3T)
    for b in range(B):
        K.gemm_bf16(rel[b * n:(b + 1) * n, :hw8], q3T[b], out_bf16=cat[b * n:(b + 1) * n, :C])
    # out3 = relu(out3_proj(cat[out2, out])) + relu(vis_4 x)  (:65-71)
    q4 = ws.get("pw_q", (N_, C), torch.float32, dev)
    K.gemm_bf16(xb, wb("v4_w", fusion.vis_4[0]), bias=b_(fusion.vis_4[0]), act=K.ACT_RELU, out_f32=q4)
    r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
    rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
    K.gemm_bf16(cat[:, :2 * C], wb("o3_w", fusion.out3_proj[0]), bias=b_(fusion.out3_proj[0]), act=K.ACT_RELU, resid=q4, out_f32=r32, out_bf16=rb)
    _count(11 + 3 * B)
    _language_gate(x, rb, res_gate, pw, q, gate_act)
    return r32


def efn_gate(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, ws: Workspace,
             gate_act: str = "tanh", r_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """EFN fusion (reference lib/bcam.py:172-269, --efn) + LanguageGate; same contract as ``pwam_gate``.  The token axis is read as a square
    image (h = sqrt(n)) and 2 x 2 pooled when n > 225, as in the reference; the co-attention maps are (n/4)^2 at most (3600^2 at 480 x 480)."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    h = int(round(n ** 0.5))
    pooled = n > 225                         # (:243)
    if h * h != n or (pooled and h % 2):
        raise K.LavtError(f"EFN: {n} tokens are not a square (even-sided when pooled) feature map (reference lib/bcam.py:239-249)")
    pw = fusion.prepared
    att = fusion.image_lang_att
    Nl = l.shape[-1]
    Nlp = (Nl + 31) // 32 * 32
    n2 = n // 4 if pooled else n             # co-attention positions
    n2p = (n2 + 31) // 32 * 32
    scale = C ** -0.5

    def cs(N):
        return pw.get("cs_%d" % N, [], lambda: torch.full((N,), scale, device=dev, dtype=torch.float32))

    # M = gelu(project(cat[x, sentence])) (:179-185): the sentence half of the Conv1d is a per-image bias
    pj = fusion.project[0]
    sb = ws.get("ef_sb", (B, C), torch.float32, dev)
    K.efn_sentence_bias(l, mask, pw.get("pj_wl", [pj.weight], lambda: _f32(pj.weight[:, C:, 0])), _f32(pj.bias), sb)
    wx = pw.get("pj_wx", [pj.weight], lambda: _bf16(pj.weight[:, :C, 0]))
    M = ws.get("pw_vis", (N_, C), torch.bfloat16, dev)
    for b in range(B):
        K.gemm_bf16(xb[b * n:(b + 1) * n], wx, bias=sb[b], act=K.ACT_GELU, out_bf16=M[b * n:(b + 1) * n])
    # lang = gelu(lang_project(l)) * mask; L = softmax(C^-0.5 M lang + pad mask) lang^T (:186-194)
    lp = fusion.lang_project[0]
    lang = ws.get("bc_lr", (B, Nlp, C), torch.bfloat16, dev)
    langT = ws.get("bc_lrT", (B, C, Nlp), torch.bfloat16, dev)
    K.bcam_words(l, pw.get("lp_w", [lp.weight], lambda: _f32(lp.weight[:, :, 0])), _f32(lp.bias), lang, langT, mask=mask, act=K.ACT_GELU)
    sim = ws.get("bc_sim", (N_, Nlp), torch.float32, dev)
    for b in range(B):
        K.gemm_bf16(M[b * n:(b + 1) * n], lang[b], cscale=cs(Nlp), out_f32=sim[b * n:(b + 1) * n])
    # f_key(L) = sum_j p_j f_key(lang_j): the key side stays fp32 up to its InstanceNorm (see csrc/bcam_kernels.cu: efn_word_attend_kernel)
    fk = att.f_key[0]
    G = ws.get("ef_G", (B, Nlp, C), torch.float32, dev)
    K.gemm_bf16(lang.view(B * Nlp, C), pw.get("fk_w", [fk.weight], lambda: _bf16(_conv1x1_w(fk))), bias=fk.bias.detach(), out_f32=G.view(B * Nlp, C))
    # EFNAttention (:236-269): q = pool(IN(f_query M)), k = pool(IN(f_key L))
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(B, n, C),), torch.float32, dev)
    stats = ws.get("pw_stats", (B, 2, C), torch.float32, dev)
    pre = ws.get("pw_q", (B, n, C), torch.float32, dev)
    qk = []
    for name in ("fq", "fk"):
        if name == "fq":
            conv = att.f_query[0]
            K.gemm_bf16(M, pw.get("fq_w", [conv.weight], lambda: _bf16(_conv1x1_w(conv))), bias=conv.bias.detach(), out_f32=pre.view(N_, C))
        else:
            K.efn_word_attend(sim, mask, G, pre.view(N_, C))
        K.instnorm_stats(pre, stats, stw)
        t = ws.get("ef_" + name, (B, n2p, C), torch.bfloat16, dev)
        K.efn_norm_pool(pre, stats, t, h, pooled)
        qk.append(t)
    q, k = qk
    qT = ws.get("ef_qT", (B, C, n2p), torch.bfloat16, dev)
    kT = ws.get("ef_kT", (B, C, n2p), torch.bfloat16, dev)
    K.bcam_transpose_pad(q.view(B * n2p, C), qT)
    K.bcam_transpose_pad(k.view(B * n2p, C), kT)
    logits = ws.get("bc_logits", (n2, n2p), torch.float32, dev)
    prob = ws.get("bc_rel", (n2, n2p), torch.bfloat16, dev)
    cat = ws.get("bc_cat", (B, n2, 2 * C), torch.bfloat16, dev)            # Lp | Mp
    for b in range(B):
        # Lp = softmax_rows(sim) k ; Mp = softmax_cols(sim)^T q = softmax_rows(sim^T) q   (:251-258)
        for a_, w_, vT, col in ((q, k, kT, 0), (k, q, qT, C)):
            K.gemm_bf16(a_[b, :n2], w_[b], cscale=cs(n2p), out_f32=logits)
            K.bcam_softmax_rows(logits, n2, prob)
            K.gemm_bf16(prob, vT[b], out_bf16=cat[b, :, col:col + C])
    # W: Conv1d(2C -> C, k = 3, pad 1) over the flattened token axis = centre tap + two row-shifted accumulations; then IN (+ upsample)
    Wc = att.W[0]
    taps = pw.get("W_taps", [Wc.weight], lambda: [_bf16(Wc.weight[:, :, t]) for t in range(3)])
    o = ws.get("pw_q", (B, n2, C), torch.float32, dev)                     # q / k pre-activations are dead
    for b in range(B):
        K.gemm_bf16(cat[b], taps[1], bias=Wc.bias.detach(), out_f32=o[b])
        K.gemm_bf16(cat[b, :n2 - 1], taps[0], resid=o[b, 1:], out_f32=o[b, 1:])          # out[i] += W[:, :, 0] cat[i - 1]
        K.gemm_bf16(cat[b, 1:], taps[2], resid=o[b, :n2 - 1], out_f32=o[b, :n2 - 1])      # out[i] += W[:, :, 2] cat[i + 1]
    K.instnorm_stats(o, stats, stw)
    r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
    rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
    K.efn_norm_upsample(o, stats, n, h, pooled, out_f32=r32, out_bf16=rb)
    _count(13 + 11 * B)
    _language_gate(x, rb, res_gate, pw, M, gate_act)
    return r32


def sep_t_pwam_gate(x: torch.Tensor, xb: torch.Tensor, fusion, res_gate, l: torch.Tensor, mask: torch.Tensor, B: int, D: int,
                    H: int, W: int, ws: Workspace, gate_act: str = "tanh", r_f32: Optional[torch.Tensor] = None) -> torch.Tensor:
    """SepTPWAM + LanguageGate under the README video flags (reference SepTPWAM.forward :1480-1584): every projection of
    ``pwam_gate`` is the sum of a Conv3d(3,3,3) branch (implicit GEMM over NDHWC with 5-D TMA boxes) and a Conv3d(1,1,1)
    branch (plain GEMM).  x fp32 [B*n, C] is updated in place with the gated residual; returns r fp32 [B*n, C]."""
    N_, C = x.shape
    n = N_ // B
    dev = x.device
    pw = fusion.prepared
    heads = fusion.num_heads
    Nl = l.shape[-1]

    def w333(name, conv):     # (Cout, Cin, kz, ky, kx) -> [Cout, ((kz*3+ky)*3+kx)*Cin + ci]
        return pw.get(name, [conv.weight], lambda: _bf16(conv.weight.detach().permute(0, 2, 3, 4, 1).reshape(conv.weight.shape[0], -1)))

    def w111(name, conv):
        return pw.get(name, [conv.weight], lambda: _bf16(conv.weight.detach().reshape(conv.weight.shape[0], -1)))

    def b_(conv):
        return conv.bias.detach()

    xb5 = xb.view(B, D, H, W, C)
    t32 = ws.get("sp_t32", (N_, C), torch.float32, dev)              # temporal-branch result waiting for the spatial one
    # ts_vis = GELU(conv333(x)) + GELU(conv111(x))                     (:1487-1503)
    vt, vs_ = fusion.temporal_vis_project[0], fusion.spatial_vis_project[0]
    K.conv3d_bf16(xb5, w333("vis_t", vt), bias=b_(vt), act=K.ACT_GELU, out_f32=t32)
    vis = ws.get("pw_vis", (B, n, C), torch.bfloat16, dev)
    K.gemm_bf16(xb, w111("vis_s", vs_), bias=b_(vs_), act=K.ACT_GELU, resid=t32, out_bf16=vis.view(N_, C))
    # query = IN3d(conv333(x)) + IN3d(conv111(x))                      (:1512-1524)
    qa = ws.get("pw_q", (B, n, C), torch.float32, dev)
    qb = ws.get("sp_qb", (B, n, C), torch.float32, dev)
    sa = ws.get("pw_stats", (B, 2, C), torch.float32, dev)
    sb = ws.get("sp_stats_b", (B, 2, C), torch.float32, dev)
    stw = ws.get("pw_statw", (K.instnorm_workspace_floats(B, n, C),), torch.float32, dev)
    qt, qs = fusion.f_query_t[0], fusion.f_query_s[0]
    K.conv3d_bf16(xb5, w333("q_t", qt), bias=b_(qt), out_f32=qa.view(N_, C))
    K.gemm_bf16(xb, w111("q_s", qs), bias=b_(qs), out_f32=qb.view(N_, C))
    K.instnorm_stats(qa, sa, stw)
    K.instnorm_stats(qb, sb, stw)
    K.instnorm_sum2(qa, sa, qb, sb, qa)
    ident = pw.get("ident_%d_%s" % (B, dev), [], lambda: torch.stack([torch.zeros(B, C), torch.ones(B, C)], 1).to(dev).contiguous())
    # words: k, v and the masked softmax are those of PWAM             (:1534-1553)
    k_w = pw.get("k_w", [fusion.f_key[0].weight], lambda: _f32(_conv1x1_w(fusion.f_key[0])))
    v_w = pw.get("v_w", [fusion.f_value[0].weight], lambda: _f32(_conv1x1_w(fusion.f_value[0])))
    kk = ws.get("pw_k", (B, Nl, C), torch.float32, dev)
    vv = ws.get("pw_v", (B, Nl, C), torch.float32, dev)
    K.pwam_kv(l, mask, k_w, b_(fusion.f_key[0]), v_w, b_(fusion.f_value[0]), kk, vv)
    o = ws.get("pw_o", (B, n, C), torch.bfloat16, dev)
    K.pwam_attend(qa, ident, kk, vv, mask, o, heads)
    # lang = IN3d(conv333(o)) + IN3d(conv111(o))                       (:1556-1561)
    Wt, Ws = fusion.W_t[0], fusion.W_s[0]
    K.conv3d_bf16(o.view(B, D, H, W, C), w333("W_t", Wt), bias=b_(Wt), out_f32=qa.view(N_, C))
    K.gemm_bf16(o.view(N_, C), w111("W_s", Ws), bias=b_(Ws), out_f32=qb.view(N_, C))
    K.instnorm_stats(qa, sa, stw)
    K.instnorm_stats(qb, sb, stw)
    K.instnorm_sum2(qa, sa, qb, sb, qa)
    a2 = o  # o is dead after the W projections
    K.pwam_mul_norm(vis, qa, ident, a2)
    # r = GELU(conv333(mm)) + GELU(conv111(mm))                         (:1574-1578)
    mt, ms = fusion.project_mm_t[0], fusion.project_mm_s[0]
    K.conv3d_bf16(a2.view(B, D, H, W, C), w333("mm_t", mt), bias=b_(mt), act=K.ACT_GELU, out_f32=t32)
    r32 = r_f32 if r_f32 is not None else ws.get("pw_r32", (N_, C), torch.float32, dev)
    rb = ws.get("pw_rb", (N_, C), torch.bfloat16, dev)
    K.gemm_bf16(a2.view(N_, C), w111("mm_s", ms), bias=b_(ms), act=K.ACT_GELU, resid=t32, out_f32=r32, out_bf16=rb)
    _count(19)
    _language_gate(x, rb, res_gate, pw, vis.view(N_, C), gate_act)      # vis is dead: scratch
    return r32


# ------------------------------------------------------------------------------------------------
# PatchMerging (reference :289-311) and PatchEmbed3D (:616-634)
# ------------------------------------------------------------------------------------------------
def patch_merging(x: torch.Tensor, ds, B: int, D: int, H: int, W: int, ws: Workspace, out: torch.Tensor) -> None:
    """x fp32 [B*D*H*W, C] -> out fp32 [B*D*ceil(H/2)*ceil(W/2), 2C]."""
    C = x.shape[1]
    dev = x.device
    H2, W2 = (H + 1) // 2, (W + 1) // 2
    red_w = ds.prepared.get("red_w", [ds.reduction.weight], lambda: _bf16(ds.reduction.weight))
    g = ws.get("merge", (B * D * H2 * W2, 4 * C), torch.bfloat16, dev)
    K.patch_merge_layernorm(x, B, D, H, W, ds.norm.weight, ds.norm.bias, g, eps=ds.norm.eps)
    K.gemm_bf16(g, red_w, out_f32=out)
    _count(2)


def patch_embed(x5: torch.Tensor, pe, ws: Workspace, out: torch.Tensor) -> Tuple[int, int]:
    """x5 fp32 (B,3,T,H,W) strided view; out fp32 [B*T*Hp*Wp, C].  Returns (Hp, Wp)."""
    B, _, T, H, W = x5.shape
    dev = x5.device
    Hp, Wp = (H + 3) // 4, (W + 3) // 4
    C = pe.embed_dim

    def _w():
        w = pe.proj.weight.detach().reshape(C, -1).to(torch.bfloat16)     # [C, 48], col = c*16 + ph*4 + pw
        wp = torch.zeros(C, 64, device=w.device, dtype=torch.bfloat16)
        wp[:, : w.shape[1]] = w
        return wp
    pw_ = pe.prepared.get("w", [pe.proj.weight], _w)
    cols = ws.get("pe_cols", (B * T * Hp * Wp, 64), torch.bfloat16, dev)
    K.patch_embed_im2col(x5, cols)
    if pe.norm is not None:
        K.gemm_bf16(cols, pw_, bias=pe.proj.bias.detach(), out_f32=out)
        K.layernorm_rows(out, pe.norm.weight, pe.norm.bias, out_f32=out, eps=pe.norm.eps)   # row-wise, safe in place
        _count(3)
    else:
        K.gemm_bf16(cols, pw_, bias=pe.proj.bias.detach(), out_f32=out)
        _count(2)
    return Hp, Wp


# ------------------------------------------------------------------------------------------------
# SimpleDecoding (reference lib/mask_predictor.py:56-99) on NHWC bf16 feature maps
# ------------------------------------------------------------------------------------------------
def _bn_fold(bn):
    s = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
    return s.contiguous(), (bn.bias.detach().float() - bn.running_mean.detach().float() * s).contiguous()


def _conv_taps(conv) -> torch.Tensor:
    w = conv.weight.detach()                                    # [Cout, Cin, 3, 3]
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).to(torch.bfloat16).contiguous()   # [(ky*3+kx)*Cin + ci]


def _upconv_bn_relu(y: torch.Tensor, skip: Optional[torch.Tensor], dec, conv_name: str, bn_name: str, ws: Workspace,
                    out: torch.Tensor) -> None:
    """out = ReLU(BN(conv3x3(cat[bilinear(y -> out size, align_corners=True), skip]))) without the upsampled map: conv and upsample are
    both linear, so the upsampled half of the conv is Z = W_tap . y on the coarse grid (one GEMM, N = 9 * hid) blended by
    upconv_blend.  At the x2 levels that is a quarter of the FLOPs of the conv over up(y).  ``skip`` None: no skip channels."""
    conv, bn = getattr(dec, conv_name), getattr(dec, bn_name)
    if bn.training:
        raise K.LavtError("SimpleDecoding on the B200 path is inference-only (BatchNorm must be in eval mode)")
    n_img, h, w, cy = y.shape
    _, H, W, hid = out.shape
    dev = y.device
    # row tap*hid + co holds w[co, :C_Y, ky, kx]
    wy = dec.prepared.get(conv_name + "_up", [conv.weight],
                          lambda: conv.weight.detach()[:, :cy].permute(2, 3, 0, 1).reshape(9 * hid, cy).to(torch.bfloat16).contiguous())
    s, b = dec.prepared.get(bn_name, [bn.weight, bn.bias, bn.running_mean, bn.running_var], lambda: _bn_fold(bn))
    z = ws.get("dec_z", (n_img, h, w, 9 * hid), torch.bfloat16, dev)
    K.gemm_bf16(y.view(-1, cy), wy, out_bf16=z.view(-1, 9 * hid))
    p = None
    if skip is not None:
        w_s = dec.prepared.get(conv_name + "_skip", [conv.weight],
                               lambda: conv.weight.detach()[:, cy:].permute(0, 2, 3, 1).reshape(hid, -1).to(torch.bfloat16).contiguous())
        p = ws.get("dec_p", (n_img, H, W, hid), torch.float32, dev)
        K.conv3x3_bf16(skip, w_s, cscale=s, bias=b, out_f32=p.view(-1, hid))
        _count(1)
    K.upconv_blend(z, p, s, b, out)
    _count(2)


def _cbr(x_nhwc: torch.Tensor, dec, conv_name: str, bn_name: str, out: torch.Tensor) -> None:
    conv, bn = getattr(dec, conv_name), getattr(dec, bn_name)
    if bn.training:
        raise K.LavtError("SimpleDecoding on the B200 path is inference-only (BatchNorm must be in eval mode)")
    w = dec.prepared.get(conv_name, [conv.weight], lambda: _conv_taps(conv))
    s, b = dec.prepared.get(bn_name, [bn.weight, bn.bias, bn.running_mean, bn.running_var], lambda: _bn_fold(bn))
    K.conv3x3_bf16(x_nhwc, w, cscale=s, bias=b, act=K.ACT_RELU, out_bf16=out.view(-1, out.shape[-1]))
    _count(1)


def decoder_nhwc(dec, c4: torch.Tensor, c3: torch.Tensor, c2: torch.Tensor, c1: torch.Tensor, ws: Workspace,
                 logits_nchw: Optional[torch.Tensor], feats: Optional[list] = None) -> torch.Tensor:
    """c_i bf16 NHWC [n_img, H_i, W_i, C_i] (c1 = None under --lazy_pred); optional logits_nchw fp32 [n_img, 2, H_1, W_1].
    Returns the low-resolution logits as an NHWC fp32 workspace view [n_img, H_1, W_1, 2].
    ``feats``: if a list, the three top-down maps after conv2_4 / conv2_3 / conv2_2 (NHWC bf16 workspace views) are
    appended (SimpleDecoding.forward_feats, lib/mask_predictor.py:102-150)."""
    dev = c4.device
    n_img = c4.shape[0]
    hid = dec.conv1_4.weight.shape[0]
    y = c4
    if (c1 is None) != bool(getattr(dec, "lazy_pred", False)):
        raise K.LavtError("decoder: the 1/4-scale map is omitted exactly when the decoder was built with --lazy_pred")
    for skip, (ca, ba, cb, bb) in ((c3, ("conv1_4", "bn1_4", "conv2_4", "bn2_4")),
                                   (c2, ("conv1_3", "bn1_3", "conv2_3", "bn2_3")),
                                   (c1, ("conv1_2", "bn1_2", "conv2_2", "bn2_2"))):
        if skip is None:                      # --lazy_pred: no 1/4-scale level (reference lib/mask_predictor.py:77)
            continue
        _, H, W, Cs = skip.shape
        if y.shape[1] > H or y.shape[2] > W:
            raise K.LavtError("decoder: coarser map is larger than the skip connection")
        t1 = ws.get("dec_t1", (n_img, H, W, hid), torch.bfloat16, dev)
        _upconv_bn_relu(y, skip, dec, ca, ba, ws, t1)
        t2 = ws.get("dec_t2_%d" % H, (n_img, H, W, hid), torch.bfloat16, dev)
        _cbr(t1, dec, cb, bb, t2)
        y = t2
        if feats is not None:
            feats.append(t2)
    if getattr(dec, "interpolate_before_seg", False):          # reference lib/mask_predictor.py:88-97
        fine = c1
        for on, (cname, bname, mul_) in ((True, ("conv2_1", "bn1_1", 2)), (getattr(dec, "seg_last", False), ("conv1_0", "bn1_0", 4))):
            if not on:
                continue
            H, W = mul_ * fine.shape[1], mul_ * fine.shape[2]
            out = ws.get("dec_y_%d" % mul_, (n_img, H, W, hid), torch.bfloat16, dev)
            _upconv_bn_relu(y, None, dec, cname, bname, ws, out)
            y = out
    _, H, W, _ = y.shape
    w11 = dec.prepared.get("w11", [dec.conv1_1.weight], lambda: _f32(dec.conv1_1.weight.reshape(2, -1)))
    lg = ws.get("dec_logits", (n_img, H, W, 2), torch.float32, dev)
    K.conv1x1_logits(y.view(-1, hid), w11, dec.conv1_1.bias.detach(), lg.view(-1, 2))
    _count(1)
    if logits_nchw is not None:
        K.upsample_logits(lg, logits_nchw)      # same size: exact NHWC -> NCHW transposition
        _count(1)
    return lg


# ------------------------------------------------------------------------------------------------
# VLT fuse-and-classify head (reference VLTFuseAndClassify.forward, lib/vlt.py:129-199, and the modules it owns)
# ------------------------------------------------------------------------------------------------
def _fold_conv_bn(conv, bn, pad_cin: int = 0):
    """Conv2d (no bias) weight as a GEMM / tap-major operand + the eval BatchNorm folded to (scale, shift)."""
    w = conv.weight.detach()
    if w.shape[-1] == 1:
        wt = w.reshape(w.shape[0], -1)
    else:                                          # [Cout, Cin, 3, 3] -> [Cout, (ky*3+kx)*Cin' + ci], input channels zero-padded to Cin'
        cin = w.shape[1] + pad_cin
        wp = torch.zeros(w.shape[0], 3, 3, cin, device=w.device, dtype=w.dtype)
        wp[..., : w.shape[1]] = w.permute(0, 2, 3, 1)
        wt = wp.reshape(w.shape[0], -1)
    s, b = _bn_fold(bn)
    return wt.to(torch.bfloat16).contiguous(), s, b


def _pad_rows(w: torch.Tensor, rows: int) -> torch.Tensor:
    out = torch.zeros(rows, w.shape[1], device=w.device, dtype=torch.bfloat16)
    out[: w.shape[0]] = w.detach()
    return out


def _mha_layer(pw: PreparedWeights, tag: str, mha, xq_b: torch.Tensor, xkv_b: torch.Tensor, B: int, ws: Workspace, key_mask=None,
               *, resid: torch.Tensor, out_f32: torch.Tensor, out_bf16: Optional[torch.Tensor] = None) -> None:
    """nn.MultiheadAttention forward on batch-major rows: xq_b bf16 [B*Lq, E], xkv_b bf16 [B*S, E]; writes resid + attention output."""
    Em = mha.embed_dim
    dev = xq_b.device
    w_in = pw.get(tag + "_win", [mha.in_proj_weight], lambda: _bf16(mha.in_proj_weight))
    b_in = pw.get(tag + "_bin", [mha.in_proj_bias], lambda: _f32(mha.in_proj_bias))
    w_out = pw.get(tag + "_wout", [mha.out_proj.weight], lambda: _bf16(mha.out_proj.weight))
    nq, nk = xq_b.shape[0], xkv_b.shape[0]
    if xq_b.data_ptr() == xkv_b.data_ptr():                 # self-attention: one packed projection
        qkv = ws.get("vlt_qkv", (nq, 3 * Em), torch.bfloat16, dev)
        K.gemm_bf16(xq_b, w_in, bias=b_in, out_bf16=qkv)
        q, k, v = qkv[:, :Em], qkv[:, Em:2 * Em], qkv[:, 2 * Em:]
        _count(1)
    else:
        qb = ws.get("vlt_q", (nq, Em), torch.bfloat16, dev)
        kv = ws.get("vlt_kv", (nk, 2 * Em), torch.bfloat16, dev)
        K.gemm_bf16(xq_b, w_in[:Em], bias=b_in[:Em], out_bf16=qb)
        K.gemm_bf16(xkv_b, w_in[Em:], bias=b_in[Em:], out_bf16=kv)
        q, k, v = qb, kv[:, :Em], kv[:, Em:]
        _count(2)
    att = ws.get("vlt_att", (nq, Em), torch.bfloat16, dev)
    K.mha_small(q, k, v, att, B, mha.num_heads, key_mask=key_mask)
    K.gemm_bf16(att, w_out, bias=mha.out_proj.bias.detach(), resid=resid, out_f32=out_f32, out_bf16=out_bf16)
    _count(2)


def _post_norm(x32: torch.Tensor, xb: torch.Tensor, ln) -> None:
    K.layernorm_rows(x32, ln.weight, ln.bias, out_f32=x32, out_bf16=xb, eps=ln.eps)     # row-wise: safe in place
    _count(1)


def _ffn_layer(pw: PreparedWeights, tag: str, layer, x32: torch.Tensor, xb: torch.Tensor, ws: Workspace) -> None:
    w1 = pw.get(tag + "_w1", [layer.linear1.weight], lambda: _bf16(layer.linear1.weight))
    w2 = pw.get(tag + "_w2", [layer.linear2.weight], lambda: _bf16(layer.linear2.weight))
    hid = ws.get("vlt_ffn", (x32.shape[0], w1.shape[0]), torch.bfloat16, x32.device)
    K.gemm_bf16(xb, w1, bias=layer.linear1.bias.detach(), act=K.ACT_RELU, out_bf16=hid)
    K.gemm_bf16(hid, w2, bias=layer.linear2.bias.detach(), resid=x32, out_f32=x32)
    _count(2)


def vlt_head(head, c4: torch.Tensor, c3: torch.Tensor, c2: torch.Tensor, l: torch.Tensor, mask: torch.Tensor, ws: Workspace) -> torch.Tensor:
    """c4 / c3 / c2 bf16 NHWC [B, s/2, s/2, 1024] / [B, s, s, 512] / [B, 2s, 2s, 256]; l fp32 [B,768,Nl]; mask fp32 [B,Nl].
    Returns the logits as an NHWC fp32 workspace view [B, 8s, 8s, 2]."""
    dev = c4.device
    pw = head.prepared
    B, s4, _, C4 = c4.shape
    s = c3.shape[1]
    if head.training:
        raise K.LavtError("the VLT head on the B200 path is inference-only (BatchNorm must be in eval mode)")
    if (s, 2 * s4, c2.shape[1]) != (head.size, s, 2 * s) or c3.shape[2] != s or (C4, c3.shape[3], c2.shape[3]) != (1024, 512, 256):
        raise K.LavtError(f"VLT head built for img_size {16 * head.size}: needs {head.size // 2}^2 x 1024, {head.size}^2 x 512 and "
                          f"{2 * head.size}^2 x 256 maps, got {tuple(c4.shape)}, {tuple(c3.shape)}, {tuple(c2.shape)}")
    P4, P3, Q, Dm = B * s4 * s4, B * s * s, head.num_queries, head.d_model
    Nl = l.shape[-1]

    def cb(tag, seq, i=0, pad_cin=0):
        return pw.get(tag, [seq[i].weight, seq[i + 1].weight, seq[i + 1].bias, seq[i + 1].running_mean, seq[i + 1].running_var],
                      lambda: _fold_conv_bn(seq[i], seq[i + 1], pad_cin))

    def conv1(x2d, tag, seq, out, i=0, **kw):              # 1x1 conv + BN + ReLU on rows
        w, sc, bi = cb(tag, seq, i)
        K.gemm_bf16(x2d, w, cscale=sc, bias=bi, act=K.ACT_RELU, out_bf16=out, **kw)
        _count(1)

    def conv3(x4d, tag, seq, out2d, i=0, pad_cin=0):       # 3x3 conv + BN + ReLU on NHWC
        w, sc, bi = cb(tag, seq, i, pad_cin)
        K.conv3x3_bf16(x4d, w, cscale=sc, bias=bi, act=K.ACT_RELU, out_bf16=out2d)
        _count(1)

    # ---- sentence vector: masked mean -> Linear -> BatchNorm1d -> ReLU  (:137-139)
    lp, bn1 = head.lang_proj[0], head.lang_proj[1]

    def _lang_fold():
        sc, sh = _bn_fold(bn1)
        return (_f32(lp.weight) * sc[:, None]).contiguous(), (_f32(lp.bias) * sc + sh).contiguous()
    lw, lb = pw.get("lang_proj", [lp.weight, lp.bias, bn1.weight, bn1.bias, bn1.running_mean, bn1.running_var], _lang_fold)
    sent = ws.get("vlt_sent", (B, C4), torch.float32, dev)
    K.efn_sentence_bias(l, mask, lw, lb, sent)
    K.rows_affine_act(sent, act=K.ACT_RELU, out_f32=sent)
    # ---- x_mm_c4 = ReLU(BN((x_c4 + bottleneck(x_c4)) * sentence))  (:140-145)
    t1 = ws.get("vlt_t1", (B, s4, s4, C4 // 2), torch.bfloat16, dev)
    conv1(c4.view(P4, C4), "vr1a", head.vis_reduce_chann_1, t1.view(P4, C4 // 2))
    y4 = ws.get("vlt_y4", (P4, C4), torch.bfloat16, dev)
    conv3(t1, "vr1b", head.vis_reduce_chann_1, y4, i=3)
    jt_s, jt_b = pw.get("jt", [head.joint_threshold[0].weight, head.joint_threshold[0].bias, head.joint_threshold[0].running_mean,
                               head.joint_threshold[0].running_var], lambda: _bn_fold(head.joint_threshold[0]))
    mm4 = ws.get("vlt_mm4", (B, s4, s4, C4), torch.bfloat16, dev)
    K.rows_affine_act(y4, add=c4.view(P4, C4), v=sent, rows_per_image=s4 * s4, s=jt_s, t=jt_b, act=K.ACT_RELU, out_bf16=mm4.view(P4, C4))
    _count(4)
    # ---- level-3 fusion.  BUF columns: temp3 | Fm_mid_query | reduced c2, so both concatenations (:155, :159) are column windows
    u1 = ws.get("vlt_u1", (B, s, s, C4 + 512), torch.bfloat16, dev)            # up(x_mm_c4) | vis_reduce_chann_2(x_c3), later | project_again(..)
    t2 = ws.get("vlt_t2", (B, s, s, 512), torch.bfloat16, dev)
    conv1(c3.view(P3, 512), "vr2", head.vis_reduce_chann_2, t2.view(P3, 512))
    K.upsample_concat(mm4, t2, u1)
    buf = ws.get("vlt_buf", (P3, 1280), torch.bfloat16, dev)
    u1r = u1.view(P3, C4 + 512)
    conv1(u1r, "f12", head.fuse_1_2, buf[:, 512:1024])
    c2p = ws.get("vlt_c2p", (B, s, s, 256), torch.bfloat16, dev)
    K.avgpool2_nhwc(c2, c2p)
    conv1(c2p.view(P3, 256), "vr3", head.vis_reduce_chann_3, buf[:, 1024:1280])
    fmq = ws.get("vlt_fmq", (B, s, s, 512), torch.bfloat16, dev)
    conv1(buf[:, 512:1280], "f23", head.fuse_2_3, fmq.view(P3, 512))
    h0 = ws.get("vlt_h0", (B, s, s, 256), torch.bfloat16, dev)
    conv1(fmq.view(P3, 512), "h23a", head.hallucinate_result_of_23, h0.view(P3, 256))
    conv3(h0, "h23b", head.hallucinate_result_of_23, buf[:, 0:512], i=3)
    conv1(buf[:, 0:1024], "pa", head.project_again, u1r[:, C4:])                # overwrites the dead vis_reduce_chann_2 columns
    f1 = ws.get("vlt_f1", (P3, Dm), torch.bfloat16, dev)
    conv1(u1r, "fa", head.fuse_again, f1)
    ftf = ws.get("vlt_ftf", (P3, Dm), torch.bfloat16, dev)
    conv1(f1, "lp", head.last_project, ftf)
    _count(2)
    # ---- query generation (:329-356)
    qg = head.query_generation
    yc = ws.get("vlt_yc", (B, s, s, 520), torch.bfloat16, dev)
    K.append_coords(fmq, yc)
    ya = ws.get("vlt_ya", (B, s, s, 512), torch.bfloat16, dev)
    yb = ws.get("vlt_yb", (B, s, s, 512), torch.bfloat16, dev)
    conv3(yc, "qg_p1a", qg.project_1, ya.view(P3, 512), i=0, pad_cin=2)
    conv3(ya, "qg_p1b", qg.project_1, yb.view(P3, 512), i=3)
    conv3(yb, "qg_p1c", qg.project_1, ya.view(P3, 512), i=6)
    w_p2 = pw.get("qg_p2", [qg.project_2.weight], lambda: _pad_rows(qg.project_2.weight.reshape(Q, -1), 32))
    y16 = ws.get("vlt_y16", (P3, 32), torch.bfloat16, dev)
    K.gemm_bf16(ya.view(P3, 512), w_p2, out_bf16=y16)
    n8 = (s * s + 7) // 8 * 8
    yT = ws.get("vlt_yT", (B, 32, n8), torch.bfloat16, dev)
    K.bcam_transpose_pad(y16, yT)

    def _wq():
        w = torch.zeros(Dm, n8, device=dev, dtype=torch.bfloat16)
        w[:, : s * s] = qg.project_query[0].weight.detach()[:, :, 0]
        return w
    w_q = pw.get("qg_pq", [qg.project_query[0].weight], _wq)
    vis32 = ws.get("vlt_vis32", (B * Q, Dm), torch.float32, dev)
    for b in range(B):
        K.gemm_bf16(yT[b, :Q], w_q, act=K.ACT_RELU, out_f32=vis32[b * Q:(b + 1) * Q])
    xq = ws.get("vlt_xq", (B * Q, Dm), torch.bfloat16, dev)
    pe_q = pw.get("qg_pe_q", [qg.pos_encoder.pe], lambda: qg.pos_encoder.table(Q))
    K.rows_add_table(vis32, pe_q, out_bf16=xq)
    w_pl = pw.get("qg_pl", [qg.project_lang[0].weight], lambda: _f32(qg.project_lang[0].weight[:, :, 0]))
    zb = pw.get("qg_zb", [], lambda: torch.zeros(Dm, device=dev, dtype=torch.float32))
    lr = ws.get("vlt_lr", (B, Nl, Dm), torch.bfloat16, dev)
    lrT = ws.get("vlt_lrT", (B, Dm, Nl), torch.bfloat16, dev)
    K.bcam_words(l, w_pl, zb, lr, lrT, act=K.ACT_RELU)
    pe_l = pw.get("qg_pe_l%d" % Nl, [qg.pos_encoder.pe], lambda: qg.pos_encoder.table(Nl))
    K.rows_add_table(lr.view(B * Nl, Dm), pe_l, out_bf16=lr.view(B * Nl, Dm))
    nd32 = ws.get("vlt_nd32", (B * Q, Dm), torch.float32, dev)
    ndb = ws.get("vlt_ndb", (B * Q, Dm), torch.bfloat16, dev)
    _mha_layer(pw, "qg_mha", qg.query_gen, xq, lr.view(B * Nl, Dm), B, ws, key_mask=mask, resid=vis32, out_f32=nd32, out_bf16=ndb)
    _count(8 + B)
    # ---- transformer encoder over the s*s memory, decoder over the 16 queries (:244-264)
    tf = head.transformer_fusion
    mem32 = ws.get("vlt_mem32", (P3, Dm), torch.float32, dev)
    memb = ws.get("vlt_memb", (P3, Dm), torch.bfloat16, dev)
    pe_m = pw.get("tf_pe_m", [tf.pos_encoder.pe], lambda: tf.pos_encoder.table(s * s))
    K.rows_add_table(ftf, pe_m, out_bf16=memb, out_f32=mem32)
    for i, layer in enumerate(tf.transformer_encoder.layers):
        _mha_layer(pw, "enc%d_sa" % i, layer.self_attn, memb, memb, B, ws, resid=mem32, out_f32=mem32)
        _post_norm(mem32, memb, layer.norm1)
        _ffn_layer(pw, "enc%d" % i, layer, mem32, memb, ws)
        _post_norm(mem32, memb, layer.norm2)
    out32 = ws.get("vlt_out32", (B * Q, Dm), torch.float32, dev)
    outb = ws.get("vlt_outb", (B * Q, Dm), torch.bfloat16, dev)
    pe_t = pw.get("tf_pe_q", [tf.pos_encoder.pe], lambda: tf.pos_encoder.table(Q))
    K.rows_add_table(nd32, pe_t, out_bf16=outb, out_f32=out32)
    for i, layer in enumerate(tf.transformer_decoder.layers):
        _mha_layer(pw, "dec%d_sa" % i, layer.self_attn, outb, outb, B, ws, resid=out32, out_f32=out32)
        _post_norm(out32, outb, layer.norm1)
        _mha_layer(pw, "dec%d_ca" % i, layer.multihead_attn, outb, memb, B, ws, resid=out32, out_f32=out32)
        _post_norm(out32, outb, layer.norm2)
        _ffn_layer(pw, "dec%d" % i, layer, out32, outb, ws)
        _post_norm(out32, outb, layer.norm3)
    _count(2)
    # ---- query balancing (:396-405) + q_to_spatial (:180-182): relu(W (g y)) = g relu(W y) because the gate is a sigmoid (> 0)
    qb = head.query_balancing
    cat2 = ws.get("vlt_cat2", (B * Q, 2 * Dm), torch.bfloat16, dev)            # y | x
    wn = pw.get("qb_wn", [qb.not_decoded_query_proj[0].weight], lambda: _bf16(qb.not_decoded_query_proj[0].weight[:, :, 0]))
    wd = pw.get("qb_wd", [qb.decoded_query_proj[0].weight], lambda: _bf16(qb.decoded_query_proj[0].weight[:, :, 0]))
    K.gemm_bf16(ndb, wn, act=K.ACT_RELU, out_bf16=cat2[:, Dm:])
    K.gemm_bf16(outb, wd, act=K.ACT_RELU, out_bf16=cat2[:, :Dm])
    g0 = pw.get("qb_g0", [qb.gate_proj[0].weight], lambda: _bf16(qb.gate_proj[0].weight[:, :, 0]))
    g2 = pw.get("qb_g2", [qb.gate_proj[2].weight], lambda: _pad_rows(qb.gate_proj[2].weight[:, :, 0], 32))
    gh = ws.get("vlt_gh", (B * Q, Dm), torch.bfloat16, dev)
    K.gemm_bf16(cat2, g0, act=K.ACT_RELU, out_bf16=gh)
    gate = ws.get("vlt_gate", (B * Q, 32), torch.float32, dev)
    K.gemm_bf16(gh, g2, act=K.ACT_SIGMOID, out_f32=gate)
    ns = (s * s + 31) // 32 * 32
    w_qs = pw.get("q2s", [head.q_to_spatial[0].weight], lambda: _pad_rows(head.q_to_spatial[0].weight[:, :, 0], ns))
    sp = ws.get("vlt_sp", (B * Q, ns), torch.float32, dev)
    K.gemm_bf16(cat2[:, :Dm], w_qs, act=K.ACT_RELU, out_f32=sp)
    qmap = ws.get("vlt_qmap", (B, s * s, Q), torch.bfloat16, dev)
    K.gate_transpose(sp[:, : s * s], gate, qmap, B)
    _count(6)
    # ---- spatial refinement + progressive decoding (:183-186, :459-485)
    dec = head.decoding
    cur = ws.get("vlt_d0", (B, s, s, Dm), torch.bfloat16, dev)
    conv3(qmap.view(B, s, s, Q), "sr", head.spatial_refine, cur.view(P3, Dm))

    def dconv(x4d, name):
        conv, bn = getattr(dec, "conv" + name), getattr(dec, "bn" + name)
        w, sc, bi = pw.get("dec" + name, [conv.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var], lambda: _fold_conv_bn(conv, bn))
        n_, H_, W_, _ = x4d.shape
        o = ws.get("vlt_dc_%s" % name, (n_, H_, W_, Dm), torch.bfloat16, dev)
        K.conv3x3_bf16(x4d, w, cscale=sc, bias=bi, act=K.ACT_RELU, out_bf16=o.view(-1, Dm))
        _count(1)
        return o
    cur = dconv(dconv(cur, "1_4"), "2_4")
    for name in ("1_3", "1_2", "1_1"):
        n_, H_, W_, _ = cur.shape
        up = ws.get("vlt_up_%s" % name, (n_, 2 * H_, 2 * W_, Dm), torch.bfloat16, dev)
        K.upsample_nhwc(cur, up)
        _count(1)
        cur = dconv(up, name)
    n_, H_, W_, _ = cur.shape
    w11 = pw.get("cls_w", [dec.classifier.weight], lambda: _f32(dec.classifier.weight.reshape(2, -1)))
    lg = ws.get("vlt_logits", (n_, H_, W_, 2), torch.float32, dev)
    K.conv1x1_logits(cur.view(-1, Dm), w11, dec.classifier.bias.detach(), lg.view(-1, 2))
    _count(1)
    return lg
