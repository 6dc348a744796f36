"""Training with 8 x 12 x 12 windows (the --window12 video model): Swin blocks whose windows hold 1152 tokens (attention backward on
attn_bwd_tc2.cu) and a full training step through ``model.train(); model(x, l, m); loss.backward()``, against autograd through the CPU
oracle with the criteria and helpers of test_backward_gpu.py."""
import os
import sys

import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import test_backward_gpu as TB  # noqa: E402  (helpers: _block_setup, _oracle_grads, check_grads, check_direction, REL_TIGHT)
from oracle import lavt_oracle as O  # noqa: E402

pytestmark = pytest.mark.gpu

W12 = (8, 12, 12)


@pytest.mark.parametrize("stage,shifted,dims", [(0, True, (1, 8, 24, 24)), (0, False, (1, 8, 24, 24)), (2, True, (1, 8, 24, 24))])
def test_swin_block_backward_w12(stage, shifted, dims):
    from lavt_rs_b200 import _cabi as K
    from lavt_rs_b200 import engine as E
    from lavt_rs_b200 import train_engine as T
    cfg, sd, bb = TB._block_setup(W12)
    B, D, H, W = dims
    C, nH = 128 * 2 ** stage, 4 * 2 ** stage
    bi = 1 if shifted else 0
    blk = bb.layers[stage].blocks[bi]
    pre = f"backbone.layers.{stage}.blocks.{bi}."
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, D, H, W, C, generator=g)
    gout = torch.randn(B, D, H, W, C, generator=g)

    def fn(sd2, xx):
        return O.swin_mlp_half(O.swin_attention_half(xx, sd2, pre, nH, W12, shifted), sd2, pre)
    (dx_ref,), pg_ref = TB._oracle_grads(fn, sd, pre, [x], gout)

    ws = E.workspace("cuda")
    grads = T.GradStore()
    xf = x.cuda().reshape(-1, C).contiguous()
    out, saved = T.swin_block_fwd(xf, blk, B, D, H, W, W12, shifted, True, ws)
    assert TB.rel_l2(out, fn(sd, x).reshape(-1, C)) < 1e-2
    geom = saved[8]
    assert geom.N == 1152 and saved[-1] is not None
    assert K.window_attention_bwd_kernel(torch.empty(nH, 23 * 23 * 15), geom) == "tc2"
    dx = T.swin_block_bwd(blk, saved, gout.cuda().reshape(-1, C).contiguous(), grads, ws)
    torch.cuda.synchronize()
    assert TB.rel_l2(dx, dx_ref.reshape(-1, C)) < TB.GRAD_L2, ("dx", TB.rel_l2(dx, dx_ref.reshape(-1, C)))
    TB.check_grads(grads.named(blk), pg_ref, f"w12 swin block stage {stage} shifted={shifted}")


def test_model_training_step_w12():
    """Video model with (8, 12, 12) windows, 8 frames of 96^2: stages 0 and 1 have windows of 1152 tokens.  Loss within 2 %, direction and
    scale of every parameter gradient and of d l_feats, and the same-branch bound of test_model_training_step."""
    from lavt_rs_b200 import training as TR
    from lavt_rs_b200 import train_engine as T
    from lavt_rs_b200.weights import load_reference_state_dict
    from lavt_rs_b200.lib.video_swin_transformer import MultiModalSwinTransformer3D
    from lavt_rs_b200.lib.mask_predictor import SimpleDecoding
    from lavt_rs_b200.lib._utils import LAVT
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=W12)
    sd = O.random_state_dict(cfg, seed=0)
    g = torch.Generator().manual_seed(31)
    for s in range(4):      # the reference zero-initialises the gates (:525-526): randomise them so that their path carries gradient
        C = 128 * 2 ** s
        for k in ("0", "2"):
            sd[f"backbone.layers.{s}.res_gate.{k}.weight"] = torch.randn(C, C, generator=g) * C ** -0.5
    bb = MultiModalSwinTransformer3D(patch_size=(1, 4, 4), embed_dim=128, depths=[2, 2, 2, 2], num_heads=[4, 8, 16, 32],
                                     window_size=W12, drop_path_rate=0.0, patch_norm=True, num_heads_fusion=[1, 1, 1, 1], args=None)
    dec = SimpleDecoding(1024, None)
    load_reference_state_dict(bb, sd, "backbone.")
    load_reference_state_dict(dec, sd, "classifier.")
    model = LAVT(bb, dec).cuda().train()
    model.video = True
    B, Tn, H, W, Nl = 1, 8, 96, 96, 12
    x = torch.randn(B, Tn, 3, H, W, generator=g)
    l = torch.randn(B, 768, Nl, generator=g)
    m = torch.ones(B, Nl)
    m[0, 8:] = 0
    target = torch.randint(0, 2, (B * Tn, H, W), generator=g)

    leaf = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in sd.items()}
    lr = l.clone().requires_grad_()
    loss_ref = O.weighted_cross_entropy(O.model_forward(leaf, cfg, x, lr, m, train_bn=True), target)
    loss_ref.backward()

    # (1) the public interface: model.train(); model(x, l, m); loss.backward()
    lt = l.cuda().requires_grad_()
    out = model(x.cuda(), lt, m.cuda())
    assert out.requires_grad
    loss = torch.nn.functional.cross_entropy(out, target.cuda(), weight=torch.tensor([0.9, 1.1], device="cuda"))
    assert abs(loss.item() - loss_ref.item()) < 2e-2 * abs(loss_ref.item()), (loss.item(), loss_ref.item())
    loss.backward()
    torch.cuda.synchronize()
    got = {n: p.grad for n, p in model.named_parameters() if p.grad is not None}
    ref = {k: v.grad for k, v in leaf.items() if v.grad is not None and not k.startswith("backbone.layers.3.res_gate")}
    TB.check_direction(got, ref, "w12 training step")
    c, ratio = TB.cos_and_ratio(lt.grad, lr.grad)
    assert c > 0.95 and 0.85 < ratio < 1.18, ("dl", c, ratio)

    # (2) same-branch bound: the oracle differentiates the ReLU branches the kernels took (see test_model_training_step)
    for p in model.parameters():
        p.grad = None
    for bn in (mm for mm in dec.modules() if isinstance(mm, torch.nn.BatchNorm2d)):
        bn.reset_running_stats()
    grads = T.GradStore()
    loss1, dl = TR.segment_forward_backward(model, x.cuda(), l.cuda(), m.cuda(), target.cuda(), grads)
    torch.cuda.synchronize()
    got1 = {}
    got1.update({"backbone." + k: v for k, v in grads.named(bb).items()})
    got1.update({"classifier." + k: v for k, v in grads.named(dec).items()})
    for bn in (mm for mm in dec.modules() if isinstance(mm, torch.nn.BatchNorm2d)):
        bn.reset_running_stats()
    with torch.no_grad():
        _, tape = TR.segment_forward(model, x.cuda(), l.cuda(), m.cuda())
    branch = {}
    for _, s1, s2 in tape["dec"][0]:
        for sv in (s1, s2):
            branch["classifier." + sv[5]] = (sv[3] > 0).permute(0, 3, 1, 2).float().cpu()
    for s, st in enumerate(tape["stages"]):
        if st[1] is not None and st[1].get("g1") is not None:
            branch[f"backbone.layers.{s}.res_gate."] = (st[1]["g1"] > 0).float().cpu()
    leaf2 = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in sd.items()}
    lr2 = l.clone().requires_grad_()
    O.RELU_BRANCH = branch
    try:
        O.weighted_cross_entropy(O.model_forward(leaf2, cfg, x, lr2, m, train_bn=True), target).backward()
    finally:
        O.RELU_BRANCH = None
    ref2 = {k: v.grad for k, v in leaf2.items() if v.grad is not None and not k.startswith("backbone.layers.3.res_gate")}
    errs = {}
    for k, r in ref2.items():
        big = max(q.float().norm().item() for q in ref2.values() if q.numel() == r.numel())
        if r.float().norm().item() < 1e-3 * big:
            continue                                    # analytically zero (shift-invariant biases): covered by check_direction above
        errs[k] = TB.rel_l2(got1[k].reshape(r.shape), r)
    errs["d l_feats"] = TB.rel_l2(dl, lr2.grad)
    worst = sorted(((e, k) for k, e in errs.items()), reverse=True)
    if os.environ.get("LAVT_TEST_VERBOSE"):
        print("[w12 same-branch gradients] worst:", worst[:10], "median", sorted(errs.values())[len(errs) // 2])
    assert worst[0][0] < TB.REL_TIGHT, f"same-branch end-to-end gradients: {worst[:6]}"
