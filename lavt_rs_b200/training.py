"""Training step of the video model on the sm_100a kernels (BASELINE config 4: fwd+bwd, gradient all-reduce over NCCL).

Mirrors the inner loop of the reference's ``train_one_epoch_*`` (train.py:330-360, 398-460):

    output = model(image, text, l_mask); loss = criterion(output, target); optimizer.zero_grad(); loss.backward()

* ``segment_forward_backward`` runs the hot path after the text encoder: forward with saved activations, the reference's
  [0.9, 1.1]-weighted cross-entropy (losses.py:7-11) and the hand-written backward, leaving fp32 gradients in a
  ``GradStore`` and returning the gradient of the language features.
* ``SegmentFunction`` exposes the same computation to autograd (``model(x, text, mask)`` in ``model.train()`` mode returns
  logits whose ``.backward()`` drives the kernels), so that the reference's training loop runs unchanged.
* ``allreduce_gradients`` is the one collective of the path: bucketed NCCL all-reduce of the parameter gradients
  (replaces DistributedDataParallel, train.py:590-593).

Stochastic depth (DropPath) runs as a per-sample scale inside the proj / fc2 GEMM epilogues.  Not implemented in training mode
(raise, no fallback): --hs / --version variants.  Every window size trains, the 8 x 12 x 12 windows of --window12 included
(attention backward of windows over ~500 tokens on the tcgen05 kernel attn_bwd_tc2.cu, with a workspace from ``engine.Workspace``).  The 2-D image models
(lavt / lavt_one) train through the same code with one frame per clip.  The text encoder's own backward runs through the stock ``transformers``
module under autograd (SURVEY.md section 8f-2 marks the text side as the next row, not the hot path).
"""
from __future__ import annotations

from typing import List, Optional, Tuple

import torch

from . import _cabi as K
from . import engine as E
from . import train_engine as T


def _check_trainable(model) -> None:
    bb = model.backbone
    for layer in bb.layers:
        if getattr(layer.fusion, "kind", "pwam") in ("gacd", "bcam", "efn"):
            raise NotImplementedError("--%s is inference-only on the B200 path" % layer.fusion.kind)
        if layer.version not in ("default", "no_gate", "none"):
            raise NotImplementedError(f"--version {layer.version} is not implemented on the B200 training path")
    lazy = any(getattr(layer, "lazy_pred", False) for layer in bb.layers)
    if tuple(bb.out_indices) != ((1, 2, 3) if lazy else (0, 1, 2, 3)):
        raise NotImplementedError("training on the B200 path needs out_indices (0, 1, 2, 3), or (1, 2, 3) with --lazy_pred")
    if lazy != bool(getattr(model.classifier, "lazy_pred", False)):
        raise NotImplementedError("--lazy_pred: backbone and decoder must both be built with the flag")


def segment_forward(model, x: torch.Tensor, l_feats: torch.Tensor, l_mask: torch.Tensor, sync_bn: bool = False, lang_ready=None):
    """Forward of the hot path with saved activations.  x (B,T,3,H,W) fp32 (video) or (B,3,H,W) (image); l_feats (B,768,Nl); l_mask (B,Nl[,1]).
    ``lang_ready``: optional CUDA event after which ``l_feats`` is valid (a text encoder running on a side stream): the stream waits for
    it right before the first fusion, i.e. the patch embedding and the Swin blocks of stage 0 run under the text encoder.
    Returns (logits fp32 (B*T,2,H,W), tape)."""
    from .lib.video_swin_transformer import _lang, _mask, _planes
    _check_trainable(model)
    E.require_cuda(x, "x")
    bb, dec = model.backbone, model.classifier
    dev = x.device
    ws = E.workspace(dev)
    l = None               # read at the first fusion (after ``lang_ready``)
    mask = _mask(l_mask)
    # video: (B,T,3,H,W) -> (B,3,T,H,W) view; image models (lavt / lavt_one): (B,3,H,W) -> one frame, windows (1,w,w) never clamped
    x5 = _planes(x).permute(0, 2, 1, 3, 4) if x.dim() == 5 else _planes(x).unsqueeze(2)
    B, _, D, H, W = x5.shape
    feat, Hc, Wc, pe_saved = T.patch_embed_fwd(x5, bb.patch_embed, ws)
    stages = []
    maps = []
    for i, layer in enumerate(bb.layers):
        C = layer.dim
        n = B * D * Hc * Wc
        xb = torch.empty(n, C, device=dev, dtype=torch.bfloat16)
        blocks = []
        for bi, blk in enumerate(layer.blocks):
            feat, sv = T.swin_block_fwd(feat, blk, B, D, Hc, Wc, layer.window_size, blk.shifted, blk.clamp_window, ws,
                                        xb_out=xb if bi == layer.depth - 1 else None)
            blocks.append(sv)
        last = layer.downsample is None
        # the last stage's gated features are unused (:570-587) unless --hs makes them the stage output (:579-587)
        gate = layer.res_gate if (layer.has_gate and (not last or layer.hs)) else None
        if l is None:
            if lang_ready is not None:
                torch.cuda.current_stream().wait_event(lang_ready)
            l = _lang(l_feats)
        if layer.sep_t_pwam:
            r32, xg, pw_saved = T.sep_t_pwam_gate_fwd(feat, xb, layer.fusion, gate, l, mask, B, D, Hc, Wc, ws,
                                                      gate_act=getattr(layer, "gate_act", "tanh"))
        else:
            r32, xg, pw_saved = T.pwam_gate_fwd(feat, xb, layer.fusion, gate, l, mask, B, ws, gate_act=getattr(layer, "gate_act", "tanh"))
        if layer.version == "no_gate" and (not last or layer.hs):       # ablation: plain residual add x' = x + r (:570-575)
            xg = torch.empty_like(r32)
            K.gate_elementwise(6, pw_saved["rb"], f=feat, f2=r32, out_f32=xg)
            E._count(1)
        # --hs: stage output = gated features instead of the residual; --lazy_pred: the features BEFORE fusion (V_i, reference :556-558),
        # stages 1-3 only (no norm0, no 1/4-scale map)
        lazy = bool(getattr(layer, "lazy_pred", False))
        out_src = ((xg if xg is not None else feat) if layer.hs else (feat if lazy else r32))
        if i in bb.out_indices:
            norm = getattr(bb, f"norm{i}")
            ob = torch.empty(B * D, Hc, Wc, C, device=dev, dtype=torch.bfloat16)
            K.layernorm_rows(out_src, norm.weight, norm.bias, out_bf16=ob.view(n, C), eps=norm.eps)
            E._count(1)
            maps.append(ob)
        else:
            maps.append(None)
        merge_saved = None
        if not last:
            src = xg if xg is not None else feat
            feat, merge_saved = T.patch_merging_fwd(src, layer.downsample, B, D, Hc, Wc, ws)
        stages.append((blocks, pw_saved, out_src, merge_saved, gate is not None, bool(layer.hs), layer.version == "no_gate" and xg is not None,
                       lazy))
        if not last:
            Hc, Wc = (Hc + 1) // 2, (Wc + 1) // 2
    c1, c2, c3, c4 = maps
    lg, dec_saved = T.decoder_fwd(dec, c4, c3, c2, c1, ws, sync_bn)
    logits = torch.empty(lg.shape[0], 2, x.shape[-2], x.shape[-1], device=dev, dtype=torch.float32)
    K.upsample_logits(lg, logits)
    E._count(1)
    tape = dict(pe=pe_saved, stages=stages, dec=dec_saved, lg_shape=tuple(lg.shape), l=l, sync_bn=sync_bn)
    return logits, tape


def segment_backward(model, tape, dlogits: torch.Tensor, grads: T.GradStore, on_ready=None, on_dl_ready=None) -> torch.Tensor:
    """dlogits fp32 (B*T,2,H,W) -> parameter gradients in ``grads``; returns the gradient of l_feats (B,768,Nl).
    ``on_ready(params)`` is called as soon as the gradients of a group of parameters are complete (decoder, then each stage from the
    last to the first, then the patch embedding) so that their all-reduce can overlap the rest of the backward (``GradReducer``).
    ``on_dl_ready(dl)`` is called as soon as the gradient of l_feats is final (after the adjoint of stage 0's fusion): the text encoder's
    backward can then run on a side stream under the backward of stage 0's Swin blocks and of the patch embedding."""
    bb, dec = model.backbone, model.classifier
    dev = dlogits.device
    ws = E.workspace(dev)
    sync_bn = tape["sync_bn"]
    dlg = torch.empty(tape["lg_shape"], device=dev, dtype=torch.float32)
    K.upsample_logits_bwd(dlogits.contiguous(), dlg)
    E._count(1)
    dcs = T.decoder_bwd(dec, tape["dec"], dlg, grads, ws, sync_bn)      # (dc4, dc3, dc2, dc1)
    if on_ready is not None:
        on_ready(list(dec.parameters()))
    dl = torch.zeros_like(tape["l"])
    dx_next: Optional[torch.Tensor] = None
    for i in range(len(bb.layers) - 1, -1, -1):
        layer = bb.layers[i]
        blocks, pw_saved, out_src, merge_saved, has_gate, hs, plain_add, lazy = tape["stages"][i]
        norm = getattr(bb, f"norm{i}", None)
        has_out = i in bb.out_indices
        dxg = None
        if merge_saved is not None:
            dxg = T.patch_merging_bwd(layer.downsample, merge_saved, dx_next, grads, ws)
        if hs:      # the stage output is the gated x': its gradient joins the one coming back through PatchMerging
            dr = None
            if dxg is None:
                dxg = torch.empty_like(out_src)
                K.layernorm_rows_bwd(out_src, dcs[3 - i], norm.weight, dxg, grads.of(norm.weight), grads.of(norm.bias), eps=norm.eps)
            else:
                K.layernorm_rows_bwd(out_src, dcs[3 - i], norm.weight, dxg, grads.of(norm.weight), grads.of(norm.bias), dres=dxg, eps=norm.eps)
        elif lazy:
            dr = None      # the stage output is V_i: its gradient joins the stream gradient AFTER the fusion's adjoint (below)
        else:
            dr = torch.empty_like(out_src)
            K.layernorm_rows_bwd(out_src, dcs[3 - i], norm.weight, dr, grads.of(norm.weight), grads.of(norm.bias), eps=norm.eps)
        E._count(1)
        if plain_add and dxg is not None:      # x' = x + r: the gradient of x' reaches r as well as x
            if dr is None:
                dr = dxg.clone()
            else:
                K.gate_elementwise(6, pw_saved["rb"], f=dr, f2=dxg, out_f32=dr)
            E._count(1)
        if dr is None and (not has_gate or dxg is None):
            dx = dxg        # --hs without a gate: x' = x and the fusion output is unused (no gradient for its parameters);
                            # --lazy_pred at the last stage: nothing downstream reads the fusion (dxg is None)
        else:
            fuse_bwd = T.sep_t_pwam_gate_bwd if layer.sep_t_pwam else T.pwam_gate_bwd
            # without a gate on this stage x feeds the next stage directly, so dxg is the residual-stream gradient itself
            dx = fuse_bwd(layer.fusion, layer.res_gate if has_gate else None, pw_saved, dr, dxg, grads, ws, dl)
        if i == 0 and on_dl_ready is not None:
            on_dl_ready(dl)
        if lazy and has_out:       # d V_i: LayerNorm adjoint of the stage output, added to the gradient that came back through the fusion
            if dx is None:
                dx = torch.empty_like(out_src)
                K.layernorm_rows_bwd(out_src, dcs[3 - i], norm.weight, dx, grads.of(norm.weight), grads.of(norm.bias), eps=norm.eps)
            else:
                K.layernorm_rows_bwd(out_src, dcs[3 - i], norm.weight, dx, grads.of(norm.weight), grads.of(norm.bias), dres=dx, eps=norm.eps)
            E._count(1)
        for bi in range(layer.depth - 1, -1, -1):
            dx = T.swin_block_bwd(layer.blocks[bi], blocks[bi], dx, grads, ws)
        dx_next = dx
        if on_ready is not None:
            on_ready(list(layer.parameters()) + (list(norm.parameters()) if norm is not None else []))
    T.patch_embed_bwd(bb.patch_embed, tape["pe"], dx_next, grads, ws)
    if on_ready is not None:
        on_ready(list(bb.patch_embed.parameters()))
    return dl


def segment_forward_backward(model, x, l_feats, l_mask, target: torch.Tensor, grads: T.GradStore, sync_bn: bool = False,
                             loss_scale: float = 1.0, on_ready=None, lang_ready=None, on_dl_ready=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """One fused fwd + loss + bwd of the hot path.  target int64 (B*T,H,W) in {0,1}.  Returns (loss as a 0-d CUDA tensor, dl_feats).
    ``lang_ready`` / ``on_dl_ready``: see ``segment_forward`` / ``segment_backward`` (``SideStreamText`` provides both)."""
    logits, tape = segment_forward(model, x, l_feats, l_mask, sync_bn, lang_ready)
    acc = torch.zeros(2, device=logits.device, dtype=torch.float32)
    K.cross_entropy(logits, target, acc, phase=0)
    dlogits = torch.empty_like(logits)
    K.cross_entropy(logits, target, acc, dlogits, gscale=loss_scale, phase=1)
    E._count(2)
    dl = segment_backward(model, tape, dlogits, grads, on_ready, on_dl_ready)
    return acc[0] / acc[1], dl


class SideStreamText:
    """The text encoder's forward and backward on a side stream around ``segment_forward_backward``.  BERT-base on a few sentences is
    ~600 tiny launches in each direction (2.5 + 3.2 ms per step even as CUDA graphs) that use a handful of SMs: the forward hides under the
    patch embedding and the Swin blocks of stage 0 (the hot path needs l_feats at the first fusion), the backward under the backward of
    stage 0's Swin blocks and of the patch embedding (d l_feats is final after the adjoint of stage 0's fusion).

        side = SideStreamText(device)
        l_feats, ready = side.forward(text_fn, ids, mask)
        loss, dl = segment_forward_backward(model, x, l_feats.detach(), mask, target, grads, lang_ready=ready, on_dl_ready=side.backward_hook())
        side.join()                      # before the optimizer / the text encoder's gradient all-reduce
    """

    def __init__(self, device):
        self.side = torch.cuda.Stream(device=device, priority=-1)      # its tiny kernels go first whenever SMs free up
        self.l_feats = None
        self._keep = []

    def forward(self, text_fn, ids, mask):
        self.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side):
            self.l_feats = text_fn(ids, mask)
            ready = torch.cuda.Event()
            ready.record(self.side)
        return self.l_feats, ready

    def backward_hook(self):
        def hook(dl):
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream())
            self.side.wait_event(ev)
            self._keep.append(dl)                 # allocated on the main stream, read on the side stream: alive until join()
            with torch.cuda.stream(self.side):
                self.l_feats.backward(dl)
        return hook

    def join(self):
        torch.cuda.current_stream().wait_stream(self.side)
        self.l_feats = None
        self._keep.clear()


class SegmentFunction(torch.autograd.Function):
    """autograd bridge: logits = SegmentFunction.apply(x, l_feats, l_mask, model, sync_bn).  backward() runs the sm_100a backward,
    ACCUMULATES the parameter gradients into ``param.grad`` as a side effect (the parameters are not autograd inputs of this
    node -- there are 450 of them and the kernels never see autograd) and returns the gradient of ``l_feats`` so that the text
    encoder's autograd graph continues."""

    @staticmethod
    def forward(ctx, x, l_feats, l_mask, model, sync_bn, anchor=None):
        # ``anchor``: any tensor with requires_grad=True.  It keeps this node in the autograd graph when neither the pixels nor the
        # language features require grad (frozen or precomputed text features): the parameters are not autograd inputs here.
        logits, tape = segment_forward(model, x.detach(), l_feats.detach(), l_mask, sync_bn)
        ctx.tape, ctx.model = tape, model
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        # gradients are produced for the backbone and the classifier only: the text encoder's ~110 M parameters get theirs from
        # autograd through d l_feats, so they need no slot (and no 440 MB memset) here
        m = ctx.model
        grads = T.GradStore(list(m.backbone.parameters()) + list(m.classifier.parameters()))
        dl = segment_backward(ctx.model, ctx.tape, dlogits.float(), grads)
        grads.finalize()
        ctx.tape = None
        return None, dl, None, None, None, None


class GradReducer:
    """Gradient all-reduce driven by ``segment_backward``'s ``on_ready`` callback (replaces DistributedDataParallel, train.py:589-592):
    each finished parameter group (decoder, stages last to first, patch embedding, text encoder) is handed to ``param.grad`` and averaged
    over the ranks IN PLACE on the contiguous slices of the GradStore's flat fp32 allocation that hold the group (``param.grad`` are views
    of it): no flatten, no copy-back, the division is NCCL's ReduceOp.AVG.  Parameters without a slot (the text encoder's, whose gradients
    come from autograd) go through one coalesced all-reduce of their own tensors.

    ``overlap=True`` (default): every group's all-reduce is launched asynchronously as soon as the group is finished, so it runs on NCCL's
    stream under the backward kernels of the earlier stages; ``wait()`` joins them before the optimizer.  ``overlap=False`` defers all
    launches to ``wait()``.  ``compress='bf16'`` halves the NVLink bytes (cast, all-reduce in bf16, cast back) at the price of two extra
    passes over the bucket and bf16 rounding of the summed gradient; off by default -- 906 MB of fp32 gradients take ~3 ms of an 80 ms step
    on NVSwitch and are hidden under the backward anyway.  With one rank everything is a no-op except the hand-over to ``param.grad``."""

    def __init__(self, overlap: bool = True, compress: Optional[str] = None):
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1) else None
        self.overlap = overlap
        self.compress = compress
        self.pending = []          # (handle or None, tensors, needs_division, bf16 staging or None)
        self._avg = None
        if self.dist is not None:
            self._avg = self.dist.ReduceOp.AVG if self.dist.get_backend() == "nccl" else None     # gloo has no AVG: SUM, then divide

    def ready(self, grads: T.GradStore):
        def _cb(params):
            done = grads.finalize(only=params)
            self.reduce(done, grads)
        return _cb

    def _launch(self, tensors, async_op: bool):
        """One all-reduce per contiguous slice (a handful per group); returns the entries to join."""
        out = []
        for t in tensors:
            if self.compress == "bf16":
                stage = t.to(torch.bfloat16)
                h = self.dist.all_reduce(stage, op=self._avg or self.dist.ReduceOp.SUM, async_op=async_op)
                out.append((h if async_op else None, t, self._avg is None, stage))
            else:
                h = self.dist.all_reduce(t, op=self._avg or self.dist.ReduceOp.SUM, async_op=async_op)
                out.append((h if async_op else None, t, self._avg is None, None))
        return out

    def reduce(self, params, grads: Optional[T.GradStore] = None) -> None:
        params = [p for p in params if p.grad is not None]
        if self.dist is None or not params:
            return
        views, loose = grads.flat_ranges(params) if grads is not None else ([], params)
        tensors = list(views) + [p.grad for p in loose]
        if self.overlap:
            self.pending += self._launch(tensors, async_op=True)
        else:
            self.pending += [("deferred", t, None, None) for t in tensors]

    def wait(self) -> None:
        if self.dist is None:
            self.pending = []
            return
        deferred = [t for h, t, _, _ in self.pending if isinstance(h, str)]
        entries = [e for e in self.pending if not isinstance(e[0], str)] + (self._launch(deferred, async_op=False) if deferred else [])
        world = self.dist.get_world_size()
        for handle, t, divide, stage in entries:
            if handle is not None:
                handle.wait()
            if stage is not None:
                t.copy_(stage)
            if divide:
                t.div_(world)
        self.pending = []


def allreduce_gradients(params: List[torch.nn.Parameter], bucket_mb: int = 64) -> None:
    """Bucketed average of ``param.grad`` over the ranks (NCCL over NVLink; replaces DDP's reducer, train.py:590-593)."""
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return
    world = dist.get_world_size()
    bucket: List[torch.Tensor] = []
    size = 0

    def flush():
        nonlocal bucket, size
        if not bucket:
            return
        flat = torch.cat([g.reshape(-1) for g in bucket])
        dist.all_reduce(flat)
        flat /= world
        off = 0
        for g in bucket:
            g.copy_(flat[off:off + g.numel()].view_as(g))
            off += g.numel()
        bucket, size = [], 0

    for p in params:
        if p.grad is None:
            continue
        bucket.append(p.grad)
        size += p.grad.numel() * p.grad.element_size()
        if size >= bucket_mb << 20:
            flush()
    flush()


def uses_sync_bn(model) -> bool:
    """True if the decoder's BatchNorm layers were converted with nn.SyncBatchNorm.convert_sync_batchnorm (train.py:589)."""
    return any(isinstance(m, torch.nn.SyncBatchNorm) for m in model.classifier.modules())


def train_forward(model, x, text, l_mask):
    """``model(x, text, l_mask)`` in training mode (reference lib/_utils.py:86-108 under autograd): the text encoder runs as the stock
    transformers module under autograd, everything after it through ``SegmentFunction``."""
    if hasattr(model, "text_encoder"):
        l_feats = model.text_encoder(text, attention_mask=l_mask)[0].permute(0, 2, 1)      # (B, 768, Nl)
    else:
        l_feats = text                                                                      # LAVT: precomputed language features
    anchor = torch.zeros((), device=x.device, requires_grad=True)
    return SegmentFunction.apply(x, l_feats, l_mask, model, uses_sync_bn(model), anchor)


class GraphedTextEncoder(torch.nn.Module):
    """The text encoder's forward AND backward as two CUDA graphs (``torch.cuda.make_graphed_callables``): BERT-base on 4 x 20
    tokens is ~600 tiny kernels in each direction, i.e. launch-bound (4.8 + 3.9 ms eager vs the GPU time of a few hundred
    microseconds).  Shapes are static per (batch, sentence length); parameters stay ordinary autograd leaves."""

    class _Wrap(torch.nn.Module):
        def __init__(self, enc):
            super().__init__()
            self.enc = enc

        def forward(self, ids, mask):
            return self.enc(ids, attention_mask=mask)[0]          # last_hidden_state (B, Nl, 768)

    def __init__(self, text_encoder, sample_ids: torch.Tensor, sample_mask: torch.Tensor):
        super().__init__()
        self.wrap = self._Wrap(text_encoder)
        self.graphed = torch.cuda.make_graphed_callables(self.wrap, (sample_ids, sample_mask))
        self.shape = tuple(sample_ids.shape)

    def forward(self, ids, mask):
        if tuple(ids.shape) != self.shape:
            raise ValueError(f"GraphedTextEncoder was captured for token ids of shape {self.shape}, got {tuple(ids.shape)}")
        return self.graphed(ids, mask).permute(0, 2, 1)           # (B, 768, Nl) = lib/_utils.py:98-100
