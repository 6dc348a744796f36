"""CPU oracle for the LAVT-RS hot path -- TEST INFRASTRUCTURE ONLY.

A plain fp32 PyTorch restatement of the reference algorithm (Yxxxb/LAVT-RS), written as functions
over a ``state_dict`` with the reference's key names.  Only ``tests/``, ``__graft_entry__.smoke()``
and ``bench.py``'s CPU-baseline / ``--impl reference`` legs may import this module; the product
path (``lavt_rs_b200``) never does and has no CPU fallback.

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so the oracle
is pinned against the reference ITSELF, imported unmodified from its checkout with the shims in
``oracle/ref_shims.py``: ``oracle/make_golden.py`` runs both on seeded inputs, asserts agreement
(tests/test_oracle_vs_reference.py does the same whenever that checkout is present) and stores
small reference outputs under ``tests/golden/`` for the GPU box, where the reference is absent.

Everything is channels-last and index-math based (no roll / partition copies) so that it doubles as
the specification of the CUDA kernels.  Citations are file:line relative to the reference root.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


# --------------------------------------------------------------------------------------------
# configuration (lib/segmentation.py:154-185 for the video model, :100-150 for the image model)
# --------------------------------------------------------------------------------------------
@dataclass
class OracleConfig:
    embed_dim: int = 128
    depths: Tuple[int, ...] = (2, 2, 18, 2)
    num_heads: Tuple[int, ...] = (4, 8, 16, 32)
    window: Tuple[int, int, int] = (8, 7, 7)     # (1, w, w) for the 2-D image backbone
    patch: Tuple[int, int, int] = (1, 4, 4)
    fusion_heads: Tuple[int, ...] = (1, 1, 1, 1)  # --mha
    clamp_window: bool = True                     # 3-D backbone clamps (get_window_size); 2-D never does
    video: bool = True
    gate_act: str = "tanh"
    lazy_pred: bool = False                       # --lazy_pred: stage outputs = features BEFORE fusion (V_i, :556-558), stages 1-3 only
                                                  # (lib/segmentation.py:184-185); the decoder stops at 1/8 scale (lib/mask_predictor.py:32,77)
    hs: bool = False                              # --hs: stage output = gated x (E_i) instead of the PWAM residual (:579-587)
    bcam: bool = False                            # --bcam (2-D image backbone, 480 x 480 inputs only): BCAM fusion of lib/bcam.py:8-75
    efn: bool = False                             # --efn (2-D image backbone): EFN fusion of lib/bcam.py:160-269 (co-attention over pooled pixels)
    gacd: bool = False                            # --gacd (2-D image backbone): GA-CD fusion of lib/bcam.py:78-127 instead of PWAM
    fuse_simple: bool = False                     # --fuse simple: LangProject (mean-pooled sentence vector) instead of pixel-word attention
    att_norm: str = "IN"                          # --att_norm_layer_type of the 2-D backbone: IN | BN | LN | none (lib/backbone.py:1297-1302)
    interpolate_before_seg: bool = False          # decoder level at 1/2 scale (lib/mask_predictor.py:40-43, 88-92)
    seg_last: bool = False                        # decoder level at full scale, no final interpolation in the video model (:45-48, 93-97)
    version: str = "default"                      # --version: default = LanguageGate; no_gate = x + r; none = x (:561-575)
    sep_t_pwam: bool = False                      # README video flags: --sep_t_pwam --conv3d_kernel_size_t 3-3-3
                                                  # --conv3d_kernel_size_s 1-1-1 --w_t3x3_s1x1 --mm_t3x3_s1x1

    @staticmethod
    def swin(swin_type: str = "base", window12: bool = False, video: bool = True, mha: str = "") -> "OracleConfig":
        dims = {"tiny": (96, (2, 2, 6, 2), (3, 6, 12, 24)), "small": (96, (2, 2, 18, 2), (3, 6, 12, 24)),
                "base": (128, (2, 2, 18, 2), (4, 8, 16, 32)), "large": (192, (2, 2, 18, 2), (6, 12, 24, 48))}[swin_type]
        w = 12 if window12 else 7
        heads = tuple(int(a) for a in mha.split("-")) if mha else (1, 1, 1, 1)
        return OracleConfig(embed_dim=dims[0], depths=dims[1], num_heads=dims[2],
                            window=(8, w, w) if video else (1, w, w), fusion_heads=heads,
                            clamp_window=video, video=video)


# --------------------------------------------------------------------------------------------
# window geometry: closed forms of get_window_size / roll / window_partition / compute_mask
# --------------------------------------------------------------------------------------------
def effective_window(size, window, shift, clamp=True):
    """lib/video_swin_transformer.py:70-83."""
    ws, ss = list(window), list(shift)
    if clamp:
        for i in range(3):
            if size[i] <= window[i]:
                ws[i], ss[i] = size[i], 0
    return tuple(ws), tuple(ss)


def _axis_region(p: Tensor, P: int, w: int, s: int) -> Tensor:
    """Region id along one axis of the SHIFTED padded grid (compute_mask, :315-328)."""
    if s == 0:
        return torch.zeros_like(p)
    return (p >= P - w).long() + (p >= P - s).long()


def window_tokens(D, H, W, ws, ss, window_cfg, device=None):
    """For every (window, token) of the padded+shifted grid: source coordinates, validity, relative
    position code and mask region id.  Returns tensors of shape (nW, N)."""
    nwd, nwh, nww = -(-D // ws[0]), -(-H // ws[1]), -(-W // ws[2])
    Dp, Hp, Wp = nwd * ws[0], nwh * ws[1], nww * ws[2]
    ar = lambda n: torch.arange(n, device=device)          # noqa: E731  (index tensors live where the activations live)
    a, b, c, td, th, tw = torch.meshgrid(ar(nwd), ar(nwh), ar(nww), ar(ws[0]), ar(ws[1]), ar(ws[2]), indexing="ij")
    pd, ph, pw = a * ws[0] + td, b * ws[1] + th, c * ws[2] + tw          # shifted-grid coordinates
    d, h, w = (pd + ss[0]) % Dp, (ph + ss[1]) % Hp, (pw + ss[2]) % Wp    # == roll(-ss) then partition (:228-234)
    valid = (d < D) & (h < H) & (w < W)                                   # pad rows are zeros AFTER norm1 (:218-224)
    src = (d * H + h) * W + w
    N = ws[0] * ws[1] * ws[2]
    nW = nwd * nwh * nww
    # relative_position_index[:N,:N] slices the table index of the CONFIGURED window (:150)
    t = (td * ws[1] + th) * ws[2] + tw
    Wd, Wh, Ww = window_cfg
    cd, ch, cw = t // (Wh * Ww), (t // Ww) % Wh, t % Ww
    code = (cd * (2 * Wh - 1) + ch) * (2 * Ww - 1) + cw
    rid = 9 * _axis_region(pd, Dp, ws[0], ss[0]) + 3 * _axis_region(ph, Hp, ws[1], ss[1]) + _axis_region(pw, Wp, ws[2], ss[2])
    rs = lambda z: z.reshape(nW, N)
    return rs(src), rs(valid), rs(code), rs(rid)


def rel_const(window_cfg) -> int:
    Wd, Wh, Ww = window_cfg
    return ((Wd - 1) * (2 * Wh - 1) + (Wh - 1)) * (2 * Ww - 1) + (Ww - 1)


# --------------------------------------------------------------------------------------------
# A1: attention half of a Swin block (forward_part1 + WindowAttention3D, :137-168, :214-248)
# --------------------------------------------------------------------------------------------
def swin_attention_half(x: Tensor, sd: Dict[str, Tensor], pre: str, num_heads: int, window, shifted: bool,
                        clamp: bool = True, return_parts: bool = False, branch_scale: Optional[Tensor] = None):
    """x (B,D,H,W,C) -> x + Attn(LN1(x)).  ``pre`` = 'backbone.layers.{s}.blocks.{i}.'"""
    B, D, H, W, C = x.shape
    shift = tuple(w // 2 for w in window) if shifted else (0, 0, 0)
    ws, ss = effective_window((D, H, W), window, shift, clamp)
    src, valid, code, rid = window_tokens(D, H, W, ws, ss, window, device=x.device)
    nW, N = src.shape
    hd = C // num_heads
    xn = F.layer_norm(x, (C,), sd[pre + "norm1.weight"], sd[pre + "norm1.bias"], 1e-5).reshape(B, D * H * W, C)
    g = xn[:, src.reshape(-1).clamp(max=D * H * W - 1)] * valid.reshape(1, -1, 1).to(x.dtype)   # (B, nW*N, C)
    g = g.reshape(B * nW, N, C)
    qkv = g @ sd[pre + "attn.qkv.weight"].t() + sd[pre + "attn.qkv.bias"]
    qkv = qkv.reshape(B * nW, N, 3, num_heads, hd).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0] * hd ** -0.5, qkv[1], qkv[2]                                    # q scaled first (:147)
    s = q @ k.transpose(-1, -2)                                                        # (B*nW, nH, N, N)
    table = sd[pre + "attn.relative_position_bias_table"]                              # (L, nH)
    idx = code[:, :, None] - code[:, None, :] + rel_const(window)                      # (nW, N, N); same for all windows
    bias = table[idx[0].reshape(-1)].reshape(N, N, num_heads).permute(2, 0, 1)
    s = s + bias.unsqueeze(0)
    if any(ss):
        m = (rid[:, :, None] != rid[:, None, :]).to(x.dtype) * -100.0                  # (nW, N, N)
        s = (s.reshape(B, nW, num_heads, N, N) + m[None, :, None]).reshape(B * nW, num_heads, N, N)
    p = s.softmax(-1)
    o = (p @ v).transpose(1, 2).reshape(B * nW, N, C)
    y = o @ sd[pre + "attn.proj.weight"].t() + sd[pre + "attn.proj.bias"]
    y = y.reshape(B, nW * N, C)
    if branch_scale is not None:       # DropPath in training (:266): per-sample 0 or 1 / keep_prob on the whole branch
        y = y * branch_scale.reshape(B, 1, 1)
    out = x.reshape(B, D * H * W, C).clone()
    vi = valid.reshape(-1)
    out[:, src.reshape(-1)[vi]] += y[:, vi]                                            # window_reverse + un-roll + crop
    out = out.reshape(B, D, H, W, C)
    if return_parts:
        return out, dict(xw=g, qkv=qkv, o=o)
    return out


# A2: MLP half (:250-251, :30-36)
def swin_mlp_half(x: Tensor, sd, pre: str, branch_scale: Optional[Tensor] = None) -> Tensor:
    C = x.shape[-1]
    h = F.layer_norm(x, (C,), sd[pre + "norm2.weight"], sd[pre + "norm2.bias"], 1e-5)
    h = F.gelu(h @ sd[pre + "mlp.fc1.weight"].t() + sd[pre + "mlp.fc1.bias"])
    y = h @ sd[pre + "mlp.fc2.weight"].t() + sd[pre + "mlp.fc2.bias"]
    if branch_scale is not None:       # DropPath (:271)
        y = y * branch_scale.reshape(-1, *([1] * (y.dim() - 1)))
    return x + y


# --------------------------------------------------------------------------------------------
# A3: PWAM + LanguageGate (:919-934, :975-1009, :519-525, :561-575; 2-D: lib/backbone.py:1265-1372)
# --------------------------------------------------------------------------------------------
def _lin1x1(t: Tensor, sd, name: str) -> Tensor:
    return t @ sd[name + ".weight"][:, :, 0].t() + sd[name + ".bias"]


def _instance_norm_tokens(t: Tensor) -> Tensor:
    """InstanceNorm1d over all tokens of a clip, per channel; biased var, eps 1e-5, no affine."""
    mu = t.mean(1, keepdim=True)
    var = t.var(1, unbiased=False, keepdim=True)
    return (t - mu) / torch.sqrt(var + 1e-5)


def lang_project(l: Tensor, l_mask: Tensor, sd, pre: str) -> Tensor:
    """LangProject (:1012-1039): masked mean of the word features -> Linear -> ReLU -> Linear.  l (B,768,Nl), l_mask (B,Nl,1) -> (B,1,C)."""
    m = l_mask.to(l.dtype).transpose(1, 2)                              # (B, 1, Nl)
    s = (l * m).sum(-1) / m.sum(-1)                                     # (B, 768)
    h = F.relu(s @ sd[pre + "project.0.weight"].t() + sd[pre + "project.0.bias"])
    return (h @ sd[pre + "project.2.weight"].t() + sd[pre + "project.2.bias"]).unsqueeze(1)


def _att_norm(t: Tensor, sd, name: str, kind: str, train: bool = False) -> Tensor:
    """The norm at index 1 of f_query / W (lib/backbone.py:1297-1316) on tokens-last tensors (B, n, C); eval mode unless ``train``
    (nn.BatchNorm1d in train(): batch statistics over all clips and tokens, biased variance)."""
    if kind == "IN":
        return _instance_norm_tokens(t)
    if kind == "BN" and train:
        mean = t.mean((0, 1))
        var = t.var((0, 1), unbiased=False)
        return (t - mean) / torch.sqrt(var + 1e-5) * sd[name + ".weight"] + sd[name + ".bias"]
    if kind == "BN":
        return (t - sd[name + ".running_mean"]) / torch.sqrt(sd[name + ".running_var"] + 1e-5) * sd[name + ".weight"] + sd[name + ".bias"]
    if kind == "LN":
        return F.layer_norm(t, (t.shape[-1],), sd[name + ".weight"], sd[name + ".bias"], 1e-5)
    return t


def pwam(x: Tensor, l: Tensor, l_mask: Tensor, sd, pre: str, heads: int = 1, return_parts: bool = False, att_norm: str = "IN",
         train_norm: bool = False):
    """x (B,n,C); l (B,768,Nl); l_mask (B,Nl,1) -> x_residual (B,n,C).  ``pre`` = 'backbone.layers.{s}.fusion.'"""
    B, n, C = x.shape
    m = l_mask.to(x.dtype)                                              # (B, Nl, 1)
    vis = F.gelu(_lin1x1(x, sd, pre + "vis_project.0"))
    a = pre + "image_lang_att."
    if a + "project.0.weight" in sd:                                    # --fuse simple (:916-917, 929-930): broadcast sentence vector
        return F.gelu(_lin1x1(vis * lang_project(l, l_mask, sd, a), sd, pre + "project_mm.0"))
    q = _att_norm(_lin1x1(x, sd, a + "f_query.0"), sd, a + "f_query.1", att_norm, train_norm)          # (B, n, C)
    lt = l.transpose(1, 2)                                              # (B, Nl, 768)
    k = _lin1x1(lt, sd, a + "f_key.0") * m                              # (B, Nl, C)
    v = _lin1x1(lt, sd, a + "f_value.0") * m
    Nl = k.shape[1]
    ch = C // heads
    qh = q.reshape(B, n, heads, ch).transpose(1, 2)                     # (B, h, n, ch)
    kh = k.reshape(B, Nl, heads, ch).transpose(1, 2)                    # channel c -> head c // ch
    vh = v.reshape(B, Nl, heads, ch).transpose(1, 2)
    s = (C ** -0.5) * (qh @ kh.transpose(-1, -2))                       # scale uses the FULL C (:999)
    s = s + (1e4 * m.transpose(1, 2) - 1e4).unsqueeze(1)                # (B,1,1,Nl): pads -> -1e4
    p = s.softmax(-1)
    o = (p @ vh).transpose(1, 2).reshape(B, n, C)
    lang = _att_norm(_lin1x1(o, sd, a + "W.0"), sd, a + "W.1", att_norm, train_norm)
    r = F.gelu(_lin1x1(vis * lang, sd, pre + "project_mm.0"))
    if return_parts:
        return r, dict(vis=vis, q=q, k=k, v=v, o=o, lang=lang)
    return r


def bcam(x: Tensor, l: Tensor, l_mask: Tensor, sd, pre: str) -> Tensor:
    """BCAM fusion (lib/bcam.py:8-75, the --bcam ablation of the 2-D backbone; from BRINet): vision-guided linguistic attention (pixel-word
    softmax without scaling, keys = values = reduced word features) followed by a language-guided visual attention whose n x n map comes
    from a Linear(dim -> hw) on tanh features -- so the module only exists for n = hw (480 x 480 inputs).  x (B,n,C) -> (B,n,C)."""
    def lin(t, name):
        return t @ sd[pre + name + ".weight"].t() + sd[pre + name + ".bias"]
    lr = lin(l.transpose(1, 2), "lang_reduce")                           # (B, Nl, C)
    m = l_mask.to(x.dtype).transpose(1, 2)                               # (B, 1, Nl)
    sim = (F.relu(lin(x, "vis_1.0")) @ lr.transpose(1, 2) + (1e4 * m - 1e4)).softmax(-1)
    out = sim @ lr                                                       # (B, n, C)
    a = torch.tanh(lin(out, "out_1") + lin(F.relu(lin(x, "vis_2.0")), "vis_2_2"))
    rel = lin(a, "a_proj").softmax(-1)                                   # (B, n, hw = n)
    out2 = rel @ F.relu(lin(x, "vis_3.0"))
    out3 = F.relu(lin(torch.cat([out2, out], -1), "out3_proj.0"))
    return out3 + F.relu(lin(x, "vis_4.0"))


def efn(x: Tensor, l: Tensor, l_mask: Tensor, sd, pre: str) -> Tensor:
    """EFN fusion (lib/bcam.py:160-269, the --efn ablation of the 2-D backbone).  M = gelu(Conv1d(cat[x, masked-mean sentence vector]));
    lang = gelu(Conv1d(l)) * mask; L = softmax_words(C^-0.5 M lang + pad mask) lang^T (:172-194).  EFNAttention (:236-269): q = IN(Conv1d(M)),
    k = IN(Conv1d(L)), both 2 x 2 average-pooled when hw > 225 (the token axis is read as a square image); sim = C^-0.5 q k^T;
    Lp = softmax_rows(sim) k, Mp = softmax_cols(sim)^T q; out = IN(Conv1d(k = 3, pad 1, over the flattened token axis)(cat[Lp, Mp])),
    bilinearly upsampled x 2 (align_corners False) when pooled.  x (B,n,C); l (B,768,Nl); l_mask (B,Nl,1) -> (B,n,C)."""
    B, n, C = x.shape
    m = l_mask.to(x.dtype)                                               # (B, Nl, 1)
    lt = l.transpose(1, 2)                                               # (B, Nl, 768)
    sent = (lt * m).sum(1, keepdim=True) / m.sum(1, keepdim=True)        # (B, 1, 768)
    M = F.gelu(_lin1x1(torch.cat([x, sent.expand(B, n, -1)], -1), sd, pre + "project.0"))
    lang = F.gelu(_lin1x1(lt, sd, pre + "lang_project.0")) * m           # (B, Nl, C)
    score = (C ** -0.5) * (M @ lang.transpose(1, 2)) + (1e4 * m.transpose(1, 2) - 1e4)
    L = score.softmax(-1) @ lang                                         # (B, n, C)
    a = pre + "image_lang_att."
    q = _instance_norm_tokens(_lin1x1(M, sd, a + "f_query.0"))
    k = _instance_norm_tokens(_lin1x1(L, sd, a + "f_key.0"))
    pooled = n > 225
    h = int(n ** 0.5)
    if pooled:
        def pool(t):
            return F.avg_pool2d(t.transpose(1, 2).reshape(B, C, h, h), 2).reshape(B, C, n // 4).transpose(1, 2)
        q, k = pool(q), pool(k)
    sim = (C ** -0.5) * (q @ k.transpose(1, 2))                          # (B, n', n')
    Lp = sim.softmax(-1) @ k
    Mp = sim.softmax(-2).transpose(1, 2) @ q
    cat = torch.cat([Lp, Mp], -1).transpose(1, 2)                        # (B, 2C, n')
    out = F.conv1d(cat, sd[a + "W.0.weight"], sd[a + "W.0.bias"], padding=1)
    out = _instance_norm_tokens(out.transpose(1, 2)).transpose(1, 2)     # (B, C, n')
    if pooled:
        out = F.interpolate(out.reshape(B, C, h // 2, h // 2), scale_factor=2, mode="bilinear").reshape(B, C, n)
    return out.transpose(1, 2)


def gacd(x: Tensor, l: Tensor, l_mask: Tensor, sd, pre: str) -> Tensor:
    """GA-CD fusion (lib/bcam.py:78-127, the --gacd ablation of the 2-D backbone): sentence vector ls = LangProject(l); xm = relu(Linear(ls * x));
    one query vector per image q = Linear(ls); collection A_c = softmax_n(q . key_c(xm) dim^-0.5), diffusion A_d = sigmoid(q . key_d(xm) dim^-0.5);
    out = xm + A_d * (A_c @ value(xm)).  x (B,n,C); l (B,768,Nl); l_mask (B,Nl,1) -> (B,n,C).  ``pre`` = 'backbone.layers.{s}.fusion.'"""
    C = x.shape[-1]

    def lin(t, name):
        return t @ sd[pre + name + ".weight"].t() + sd[pre + name + ".bias"]
    ls = lang_project(l, l_mask, sd, pre + "lang_gen.")                # (B, 1, C)
    xm = F.relu(lin(ls * x, "mm_gen.0"))                                # (B, n, C)
    q = lin(ls, "query")                                                # (B, 1, C)
    a_c = (q @ lin(xm, "key_c").transpose(1, 2) * C ** -0.5).softmax(-1)           # (B, 1, n)
    a_d = torch.sigmoid(q @ lin(xm, "key_d").transpose(1, 2) * C ** -0.5)          # (B, 1, n)
    f_col = a_c @ lin(xm, "value")                                      # (B, 1, C)
    return xm + a_d.transpose(1, 2) @ f_col


# A7: SepTPWAM under the README video flags (lib/video_swin_transformer.py:1300-1584, forward :1480-1584):
# every projection of PWAM becomes the SUM of a temporal Conv3d(3,3,3) branch and a spatial Conv3d(1,1,1) branch;
# the query / W branches are each InstanceNorm3d-normalised BEFORE the sum, the vis / project_mm branches GELU'd before it.
def _conv3d_cl(x: Tensor, sd, name: str) -> Tensor:
    """x (B,D,H,W,Cin) channels-last; Conv3d weight (Cout,Cin,kd,kh,kw), stride 1, 'same' zero padding."""
    w, b = sd[name + ".weight"], sd[name + ".bias"]
    pad = tuple(k // 2 for k in w.shape[2:])
    return F.conv3d(x.permute(0, 4, 1, 2, 3), w, b, padding=pad).permute(0, 2, 3, 4, 1)


def _instance_norm_3d(t: Tensor) -> Tensor:
    """InstanceNorm3d on channels-last (B,D,H,W,C): per (clip, channel) over D*H*W; biased var, eps 1e-5, no affine."""
    B, D, H, W, C = t.shape
    return _instance_norm_tokens(t.reshape(B, D * H * W, C)).reshape(B, D, H, W, C)


def sep_t_pwam(x: Tensor, l: Tensor, l_mask: Tensor, sd, pre: str, heads: int = 1) -> Tensor:
    """x (B,D,H,W,C); l (B,768,Nl); l_mask (B,Nl,1) -> x_residual (B,D*H*W,C).  ``pre`` = 'backbone.layers.{s}.fusion.'"""
    B, D, H, W, C = x.shape
    n = D * H * W
    m = l_mask.to(x.dtype)
    vis = F.gelu(_conv3d_cl(x, sd, pre + "temporal_vis_project.0")) + F.gelu(_conv3d_cl(x, sd, pre + "spatial_vis_project.0"))  # :1487-1503
    q = _instance_norm_3d(_conv3d_cl(x, sd, pre + "f_query_t.0")) + _instance_norm_3d(_conv3d_cl(x, sd, pre + "f_query_s.0"))    # :1512-1524
    q = q.reshape(B, n, C)
    lt = l.transpose(1, 2)
    k = _lin1x1(lt, sd, pre + "f_key.0") * m                                                                                 # :1534-1538
    v = _lin1x1(lt, sd, pre + "f_value.0") * m
    Nl = k.shape[1]
    ch = C // heads
    qh = q.reshape(B, n, heads, ch).transpose(1, 2)
    kh = k.reshape(B, Nl, heads, ch).transpose(1, 2)
    vh = v.reshape(B, Nl, heads, ch).transpose(1, 2)
    s = (C ** -0.5) * (qh @ kh.transpose(-1, -2)) + (1e4 * m.transpose(1, 2) - 1e4).unsqueeze(1)                              # :1549-1552
    o = (s.softmax(-1) @ vh).transpose(1, 2).reshape(B, D, H, W, C)
    lang = _instance_norm_3d(_conv3d_cl(o, sd, pre + "W_t.0")) + _instance_norm_3d(_conv3d_cl(o, sd, pre + "W_s.0"))          # :1556-1561
    mm = vis * lang
    r = F.gelu(_conv3d_cl(mm, sd, pre + "project_mm_t.0")) + F.gelu(_conv3d_cl(mm, sd, pre + "project_mm_s.0"))               # :1574-1578
    return r.reshape(B, n, C)


# Gradient tests only: a ReLU network's gradient is discontinuous in its inputs, so an end-to-end gradient comparison is only tight when
# both sides differentiate the SAME linear branch.  RELU_BRANCH maps a ReLU site ('classifier.conv1_4', 'backbone.layers.0.res_gate.') to
# the 0/1 mask the implementation under test used in its forward; the oracle then computes x * mask there instead of relu(x).
RELU_BRANCH: Optional[Dict[str, Tensor]] = None


def _relu_site(x: Tensor, site: str) -> Tensor:
    if RELU_BRANCH is not None and site in RELU_BRANCH:
        return x * RELU_BRANCH[site].to(x.dtype).reshape(x.shape)
    return F.relu(x)


def language_gate(x: Tensor, r: Tensor, sd, pre: str, act: str = "tanh") -> Tensor:
    """x + act(W2 relu(W1 r)) * r, no biases.  ``pre`` = 'backbone.layers.{s}.res_gate.'"""
    g = _relu_site(r @ sd[pre + "0.weight"].t(), pre) @ sd[pre + "2.weight"].t()
    g = torch.tanh(g) if act == "tanh" else torch.sigmoid(g)
    return x + g * r


# A4: PatchMerging (:289-311; 2-D lib/backbone.py:261-288)
def patch_merging(x: Tensor, sd, pre: str) -> Tensor:
    """x (B,D,H,W,C) -> (B,D,ceil(H/2),ceil(W/2),2C).  ``pre`` = 'backbone.layers.{s}.downsample.'"""
    B, D, H, W, C = x.shape
    if H % 2 or W % 2:
        x = F.pad(x, (0, 0, 0, W % 2, 0, H % 2))
    parts = [x[:, :, 0::2, 0::2], x[:, :, 1::2, 0::2], x[:, :, 0::2, 1::2], x[:, :, 1::2, 1::2]]
    y = torch.cat(parts, -1)
    y = F.layer_norm(y, (4 * C,), sd[pre + "norm.weight"], sd[pre + "norm.bias"], 1e-5)
    return y @ sd[pre + "reduction.weight"].t()


# patch embedding (:616-634; 2-D lib/backbone.py:315-331): conv k=s=patch == GEMM over K=3*ph*pw, then LN
def patch_embed(x: Tensor, sd, patch) -> Tensor:
    """x (B,3,T,H,W) -> (B,T,H/4,W/4,C) channels-last."""
    B, Cin, T, H, W = x.shape
    pt, ph, pw = patch
    assert pt == 1
    if W % pw or H % ph:
        x = F.pad(x, (0, (-W) % pw, 0, (-H) % ph))
        H, W = x.shape[-2:]
    wgt = sd["backbone.patch_embed.proj.weight"]
    Cout = wgt.shape[0]
    cols = x.reshape(B, Cin, T, H // ph, ph, W // pw, pw).permute(0, 2, 3, 5, 1, 4, 6).reshape(B, T, H // ph, W // pw, Cin * ph * pw)
    y = cols @ wgt.reshape(Cout, -1).t() + sd["backbone.patch_embed.proj.bias"]
    return F.layer_norm(y, (Cout,), sd["backbone.patch_embed.norm.weight"], sd["backbone.patch_embed.norm.bias"], 1e-5)


# --------------------------------------------------------------------------------------------
# backbone forward (:854-881 with MMBasicLayer.forward :538-592) -- default flags
# --------------------------------------------------------------------------------------------
def backbone_forward(sd, cfg: OracleConfig, x: Tensor, l: Tensor, l_mask: Tensor, capture: Optional[dict] = None):
    """x (B,3,T,H,W) [video] or (B,3,H,W) [image]; l (B,768,Nl); l_mask (B,Nl,1).
    Returns the 4 stage outputs as (B*T, C_i, H_i, W_i) NCHW."""
    if x.dim() == 4:
        x = x.unsqueeze(2)
    x = patch_embed(x, sd, cfg.patch)
    if capture is not None:
        capture["patch_embed"] = x
    outs = []
    for s, depth in enumerate(cfg.depths):
        pre = f"backbone.layers.{s}."
        for i in range(depth):
            bp = f"{pre}blocks.{i}."
            x = swin_attention_half(x, sd, bp, cfg.num_heads[s], cfg.window, shifted=(i % 2 == 1), clamp=cfg.clamp_window)
            x = swin_mlp_half(x, sd, bp)
            if capture is not None:
                capture[f"s{s}b{i}"] = x
        B, D, H, W, C = x.shape
        x_pre = x                                                          # V_i (:556-558)
        if cfg.version == "swin":                                          # plain Swin stage (lib/backbone.py BasicLayer :1409-1510): no fusion
            r = None
        elif cfg.bcam:
            r = bcam(x.reshape(B, D * H * W, C), l, l_mask, sd, pre + "fusion.")
        elif cfg.gacd:
            r = gacd(x.reshape(B, D * H * W, C), l, l_mask, sd, pre + "fusion.")
        elif cfg.efn:
            r = efn(x.reshape(B, D * H * W, C), l, l_mask, sd, pre + "fusion.")
        elif cfg.sep_t_pwam:
            r = sep_t_pwam(x, l, l_mask, sd, pre + "fusion.", cfg.fusion_heads[s])
        else:
            r = pwam(x.reshape(B, D * H * W, C), l, l_mask, sd, pre + "fusion.", cfg.fusion_heads[s], att_norm=cfg.att_norm)
        if capture is not None:
            capture[f"s{s}.residual"] = r
        if cfg.version == "swin":
            pass
        elif cfg.version == "no_gate":
            x = x + r.reshape(B, D, H, W, C)
        elif cfg.version == "default" and pre + "res_gate.0.weight" in sd:
            x = language_gate(x.reshape(B, D * H * W, C), r, sd, pre + "res_gate.", cfg.gate_act).reshape(B, D, H, W, C)
        stage_out = x if (cfg.hs or cfg.version == "swin") else (x_pre if cfg.lazy_pred else r.reshape(B, D, H, W, C))   # (:579-587)
        if f"backbone.norm{s}.weight" in sd:                               # out_indices (lazy_pred: 1, 2, 3)
            o = F.layer_norm(stage_out, (C,), sd[f"backbone.norm{s}.weight"], sd[f"backbone.norm{s}.bias"], 1e-5)
            outs.append(o.permute(0, 1, 4, 2, 3).reshape(B * D, C, H, W))      # (:869-874)
        if pre + "downsample.reduction.weight" in sd:
            x = patch_merging(x, sd, pre + "downsample.")
            if capture is not None:
                capture[f"s{s}.merged"] = x
    return tuple(outs)


# --------------------------------------------------------------------------------------------
# A6: SimpleDecoding (lib/mask_predictor.py:56-99), eval-mode BatchNorm
# --------------------------------------------------------------------------------------------
def _q_bf16(t: Tensor) -> Tensor:
    """Straight-through bf16 rounding (forward: round to bf16; backward: identity).  Used ONLY by the gradient-parity tests: the
    gradient of a ReLU network is discontinuous in its inputs (an operand error of relative size eps flips ~eps of the ReLU masks and
    moves the gradient by ~sqrt(eps) in rel-L2), so a bf16 kernel can only be compared with an oracle that rounds the operands of
    the ReLU-producing contractions at the same points (conv inputs / weights are bf16 in the kernels, accumulation is fp32)."""
    return t + (t.to(torch.bfloat16).to(t.dtype) - t).detach()


def _cbr(x: Tensor, sd, conv: str, bn: str, train_bn: bool = False, emulate_bf16: bool = False) -> Tensor:
    w = sd[f"classifier.{conv}.weight"]
    if emulate_bf16:
        x, w = _q_bf16(x), _q_bf16(w)
    x = F.conv2d(x, w, padding=1)
    if train_bn:     # model.train(): batch statistics (the running buffers are updated on clones: the oracle stays functional)
        x = F.batch_norm(x, sd[f"classifier.{bn}.running_mean"].clone(), sd[f"classifier.{bn}.running_var"].clone(),
                         sd[f"classifier.{bn}.weight"], sd[f"classifier.{bn}.bias"], True, 0.1, 1e-5)
    else:
        x = F.batch_norm(x, sd[f"classifier.{bn}.running_mean"], sd[f"classifier.{bn}.running_var"],
                         sd[f"classifier.{bn}.weight"], sd[f"classifier.{bn}.bias"], False, 0.0, 1e-5)
    return _relu_site(x, f"classifier.{conv}")


def _up_to(x: Tensor, ref: Tensor) -> Tensor:
    if x.shape[-2] < ref.shape[-2] or x.shape[-1] < ref.shape[-1]:
        x = F.interpolate(x, size=ref.shape[-2:], mode="bilinear", align_corners=True)
    return x


def decoder_forward(sd, x_c4, x_c3, x_c2, x_c1, capture: Optional[dict] = None, train_bn: bool = False,
                    emulate_bf16: bool = False) -> Tensor:
    tb, eb = train_bn, emulate_bf16
    q = _q_bf16 if eb else (lambda t: t)      # the kernels hand bf16 maps from level to level
    y = torch.cat([_up_to(x_c4, x_c3), x_c3], 1)
    y = q(_cbr(_cbr(y, sd, "conv1_4", "bn1_4", tb, eb), sd, "conv2_4", "bn2_4", tb, eb))
    y = torch.cat([_up_to(y, x_c2), x_c2], 1)
    y = q(_cbr(_cbr(y, sd, "conv1_3", "bn1_3", tb, eb), sd, "conv2_3", "bn2_3", tb, eb))
    if x_c1 is not None:                       # --lazy_pred stops at 1/8 scale (lib/mask_predictor.py:77)
        y = torch.cat([_up_to(y, x_c1), x_c1], 1)
        y = q(_cbr(_cbr(y, sd, "conv1_2", "bn1_2", tb, eb), sd, "conv2_2", "bn2_2", tb, eb))
    if "classifier.conv2_1.weight" in sd:      # --interpolate_before_seg (lib/mask_predictor.py:88-92); conv2_1 is normalised by bn1_1
        y = F.interpolate(y, size=(2 * x_c1.shape[-2], 2 * x_c1.shape[-1]), mode="bilinear", align_corners=True)
        y = q(_cbr(y, sd, "conv2_1", "bn1_1", tb, eb))
        if "classifier.conv1_0.weight" in sd:  # --seg_last (:93-97)
            y = F.interpolate(y, size=(4 * x_c1.shape[-2], 4 * x_c1.shape[-1]), mode="bilinear", align_corners=True)
            y = q(_cbr(y, sd, "conv1_0", "bn1_0", tb, eb))
    if capture is not None:
        capture["dec_feat"] = y
    return F.conv2d(y, sd["classifier.conv1_1.weight"], sd["classifier.conv1_1.bias"])


def weighted_cross_entropy(logits: Tensor, target: Tensor) -> Tensor:
    """losses.py:7-11: F.cross_entropy with class weights [0.9, 1.1] (mean normalised by the summed weights)."""
    return F.cross_entropy(logits, target, weight=torch.tensor([0.9, 1.1], dtype=logits.dtype, device=logits.device))


def model_forward(sd, cfg: OracleConfig, x: Tensor, l_feats: Tensor, l_mask: Tensor, capture: Optional[dict] = None,
                  train_bn: bool = False) -> Tensor:
    """LAVTVideo.forward / LAVTOne.forward minus the (external) BERT call (lib/_utils.py:86-108, 42-63).
    x (B,T,3,H,W) for video, (B,3,H,W) for image; l_feats (B,768,Nl); l_mask (B,Nl) -> logits (B*T,2,H,W)."""
    if cfg.video:
        x = x.permute(0, 2, 1, 3, 4)
    size = x.shape[-2:]
    feats = backbone_forward(sd, cfg, x, l_feats, l_mask.unsqueeze(-1), capture)
    c1, c2, c3, c4 = feats if len(feats) == 4 else (None, *feats)        # lib/_utils.py:55-59, 101-105
    if capture is not None:
        capture.update(c1=c1, c2=c2, c3=c3, c4=c4)
    logits = decoder_forward(sd, c4, c3, c2, c1, capture, train_bn)
    if capture is not None:
        capture["logits_lowres"] = logits
    if cfg.seg_last and cfg.video:             # lib/_utils.py:105-106: the video model returns the classifier's own resolution
        return logits
    return F.interpolate(logits, size=size, mode="bilinear", align_corners=True)


# --------------------------------------------------------------------------------------------
# random-init state dict with the reference's key names and init rules (no reference import needed)
# (lib/video_swin_transformer.py:811-852: trunc_normal(.02) on Linear, zero bias, LN 1/0; Conv default init)
# --------------------------------------------------------------------------------------------
def random_state_dict(cfg: OracleConfig, seed: int = 0, l_in: int = 768) -> Dict[str, Tensor]:
    g = torch.Generator().manual_seed(seed)
    sd: Dict[str, Tensor] = {}

    def tn(*shape, std=0.02):
        return torch.nn.init.trunc_normal_(torch.empty(*shape), std=std, generator=g)

    def conv_default(*shape):
        fan_in = math.prod(shape[1:])
        b = 1.0 / math.sqrt(fan_in)
        return (torch.rand(*shape, generator=g) * 2 - 1) * b, (torch.rand(shape[0], generator=g) * 2 - 1) * b

    def ln(name, c):
        sd[name + ".weight"] = torch.ones(c) + 0.1 * torch.randn(c, generator=g)   # non-trivial affine for tests
        sd[name + ".bias"] = 0.1 * torch.randn(c, generator=g)

    C0 = cfg.embed_dim
    pe_shape = (C0, 3, *cfg.patch) if cfg.video else (C0, 3, cfg.patch[1], cfg.patch[2])
    w, b = conv_default(*pe_shape)
    sd["backbone.patch_embed.proj.weight"], sd["backbone.patch_embed.proj.bias"] = w, b
    ln("backbone.patch_embed.norm", C0)
    Wd, Wh, Ww = cfg.window
    for s, depth in enumerate(cfg.depths):
        C, nH = C0 * 2 ** s, cfg.num_heads[s]
        pre = f"backbone.layers.{s}."
        for i in range(depth):
            bp = f"{pre}blocks.{i}."
            ln(bp + "norm1", C)
            ln(bp + "norm2", C)
            sd[bp + "attn.relative_position_bias_table"] = tn((2 * Wd - 1) * (2 * Wh - 1) * (2 * Ww - 1), nH, std=0.5)
            sd[bp + "attn.qkv.weight"], sd[bp + "attn.qkv.bias"] = tn(3 * C, C, std=0.05), 0.1 * torch.randn(3 * C, generator=g)
            sd[bp + "attn.proj.weight"], sd[bp + "attn.proj.bias"] = tn(C, C), 0.02 * torch.randn(C, generator=g)
            sd[bp + "mlp.fc1.weight"], sd[bp + "mlp.fc1.bias"] = tn(4 * C, C), 0.02 * torch.randn(4 * C, generator=g)
            sd[bp + "mlp.fc2.weight"], sd[bp + "mlp.fc2.bias"] = tn(C, 4 * C), 0.02 * torch.randn(C, generator=g)
        if cfg.sep_t_pwam:
            for name in ("temporal_vis_project.0", "f_query_t.0", "W_t.0", "project_mm_t.0"):
                w, b = conv_default(C, C, 3, 3, 3)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
            for name in ("spatial_vis_project.0", "f_query_s.0", "W_s.0", "project_mm_s.0"):
                w, b = conv_default(C, C, 1, 1, 1)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
            for name in ("f_key.0", "f_value.0"):
                w, b = conv_default(C, l_in, 1)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
        elif cfg.bcam:
            hw = {128: 120 * 120, 256: 60 * 60, 512: 30 * 30, 1024: 15 * 15}[C]          # lib/bcam.py:12-19
            for name, cout, cin in (("lang_reduce", C, l_in), ("vis_1.0", C, C), ("vis_2.0", C, C), ("vis_3.0", C, C), ("vis_4.0", C, C),
                                    ("out_1", C, C), ("vis_2_2", C, C), ("a_proj", hw, C), ("out3_proj.0", C, 2 * C)):
                w, b = conv_default(cout, cin)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
        elif cfg.gacd:
            for name, cin in (("lang_gen.project.0", l_in), ("lang_gen.project.2", C), ("mm_gen.0", C), ("query", C), ("key_c", C), ("key_d", C),
                              ("value", C)):
                w, b = conv_default(C, cin)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
        elif cfg.efn:
            for name, shape in (("project.0", (C, C + l_in, 1)), ("lang_project.0", (C, l_in, 1)), ("image_lang_att.f_key.0", (C, C, 1)),
                                ("image_lang_att.f_query.0", (C, C, 1)), ("image_lang_att.W.0", (C, 2 * C, 3))):
                w, b = conv_default(*shape)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
        elif cfg.fuse_simple:
            for name in ("vis_project.0", "project_mm.0"):
                w, b = conv_default(C, C, 1)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
            for name, cin in (("project.0", l_in), ("project.2", C)):
                w, b = conv_default(C, cin)
                sd[f"{pre}fusion.image_lang_att.{name}.weight"], sd[f"{pre}fusion.image_lang_att.{name}.bias"] = w, b
        else:
            for name, cin in (("vis_project.0", C), ("image_lang_att.f_key.0", l_in), ("image_lang_att.f_query.0", C),
                              ("image_lang_att.f_value.0", l_in), ("image_lang_att.W.0", C), ("project_mm.0", C)):
                w, b = conv_default(C, cin, 1)
                sd[f"{pre}fusion.{name}.weight"], sd[f"{pre}fusion.{name}.bias"] = w, b
            if cfg.att_norm in ("BN", "LN"):            # drawn only for these variants: every other configuration keeps its random stream
                for name in ("image_lang_att.f_query.1", "image_lang_att.W.1"):
                    ln(f"{pre}fusion.{name}", C)
                    if cfg.att_norm == "BN":
                        sd[f"{pre}fusion.{name}.running_mean"] = 0.1 * torch.randn(C, generator=g)
                        sd[f"{pre}fusion.{name}.running_var"] = 1 + 0.2 * torch.rand(C, generator=g)
        sd[pre + "res_gate.0.weight"], sd[pre + "res_gate.2.weight"] = tn(C, C), tn(C, C)
        if s < len(cfg.depths) - 1:
            sd[pre + "downsample.reduction.weight"] = tn(2 * C, 4 * C)
            ln(pre + "downsample.norm", 4 * C)
        if s > 0 or not cfg.lazy_pred:
            ln(f"backbone.norm{s}", C)
    hid = 8 * C0 // 2
    levels = (("1_4", 8 * C0 + 4 * C0), ("2_4", hid), ("1_3", hid + 2 * C0), ("2_3", hid), ("1_2", hid + C0), ("2_2", hid))
    for name, cin in (levels[:4] if cfg.lazy_pred else levels):
        sd[f"classifier.conv{name}.weight"] = conv_default(hid, cin, 3, 3)[0]
        sd[f"classifier.bn{name}.weight"] = 1 + 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.bn{name}.bias"] = 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.bn{name}.running_mean"] = 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.bn{name}.running_var"] = 1 + 0.2 * torch.rand(hid, generator=g)
    w, b = conv_default(2, hid, 1, 1)
    sd["classifier.conv1_1.weight"], sd["classifier.conv1_1.bias"] = w, b
    extra = ([("conv2_1", "bn1_1")] if cfg.interpolate_before_seg else []) + ([("conv1_0", "bn1_0")] if cfg.seg_last else [])
    for cname, bname in extra:                        # drawn last: the other configurations keep their random stream
        sd[f"classifier.{cname}.weight"] = conv_default(hid, hid, 3, 3)[0]
        sd[f"classifier.{bname}.weight"] = 1 + 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.{bname}.bias"] = 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.{bname}.running_mean"] = 0.1 * torch.randn(hid, generator=g)
        sd[f"classifier.{bname}.running_var"] = 1 + 0.2 * torch.rand(hid, generator=g)
    return sd


def synthetic_inputs(B: int, T: int, H: int, W: int, Nl: int = 20, seed: int = 1, video: bool = True):
    """SURVEY.md section 8d: randn pixels, randn language features, first ceil(0.7 Nl) words valid."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T, 3, H, W, generator=g) if video else torch.randn(B, 3, H, W, generator=g)
    l = torch.randn(B, 768, Nl, generator=g)
    m = torch.zeros(B, Nl, dtype=torch.int64)
    m[:, : math.ceil(0.7 * Nl)] = 1
    return x, l, m
