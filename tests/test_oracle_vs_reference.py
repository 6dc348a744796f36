"""Pin the oracle (oracle/lavt_oracle.py) against the UNMODIFIED reference modules, imported from a
checkout of the reference (oracle/_ref or $LAVT_REFERENCE_ROOT, see oracle/ref_shims.py) with external
shims.  Runs only where that checkout exists; elsewhere the pinning of the forward and training step
is carried by tests/golden (see test_oracle_golden.py)."""
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import lavt_oracle as O  # noqa: E402
from oracle import ref_shims  # noqa: E402

pytestmark = pytest.mark.skipif(not ref_shims.reference_available(), reason="reference tree not present")


def _sd(bb, dec):
    sd = {"backbone." + k: v.detach() for k, v in bb.state_dict().items()}
    sd.update({"classifier." + k: v.detach() for k, v in dec.state_dict().items()})
    return sd


def _randomise_norms(mods, seed=3):
    """init_weights leaves LN/BN at identity; perturb them so affine / running stats are exercised."""
    g = torch.Generator().manual_seed(seed)
    for mod in mods:
        for m in mod.modules():
            if isinstance(m, (torch.nn.LayerNorm, torch.nn.BatchNorm2d)):
                m.weight.data.add_(0.1 * torch.randn(m.weight.shape, generator=g))
                m.bias.data.add_(0.1 * torch.randn(m.bias.shape, generator=g))
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.add_(0.1 * torch.randn(m.running_mean.shape, generator=g))
                m.running_var.add_(0.2 * torch.rand(m.running_var.shape, generator=g))
            if isinstance(m, torch.nn.Linear) and m.bias is not None:
                m.bias.data.add_(0.05 * torch.randn(m.bias.shape, generator=g))


@pytest.mark.parametrize("window,T,HW,mha", [((8, 7, 7), 4, (64, 64), (1, 1, 1, 1)),
                                             ((8, 7, 7), 16, (48, 40), (1, 1, 1, 1)),
                                             ((8, 12, 12), 8, (96, 96), (1, 2, 4, 4)),
                                             ((8, 12, 12), 2, (40, 52), (1, 1, 1, 1))])
def test_backbone_and_decoder_match_reference(window, T, HW, mha):
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=window, mha=mha, depths=(2, 2, 2, 2))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=window, fusion_heads=mha)
    x, l, m = O.synthetic_inputs(2, T, HW[0], HW[1], Nl=11)
    xv = x.permute(0, 2, 1, 3, 4)
    with torch.no_grad():
        ref = bb(xv, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, xv, l, m.unsqueeze(-1))
        for i, (a, b) in enumerate(zip(got, ref)):
            assert a.shape == b.shape
            err = (a - b).abs().max().item()
            assert err < 2e-4, f"stage {i}: max err {err}"
        ref_logits = dec(ref[3], ref[2], ref[1], ref[0])
        got_logits = O.decoder_forward(sd, got[3], got[2], got[1], got[0])
        assert (ref_logits - got_logits).abs().max().item() < 2e-4


@pytest.mark.parametrize("window,T,HW,mha", [((8, 7, 7), 4, (64, 64), (1, 1, 1, 1)), ((8, 7, 7), 8, (48, 40), (1, 2, 2, 4))])
def test_sep_t_pwam_backbone_matches_reference(window, T, HW, mha):
    """README video configuration: --sep_t_pwam --conv3d_kernel_size_t 3-3-3 --conv3d_kernel_size_s 1-1-1 --w_t3x3_s1x1
    --mm_t3x3_s1x1 (SepTPWAM, lib/video_swin_transformer.py:1300-1584)."""
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=window, mha=mha, depths=(2, 2, 2, 2), extra=ref_shims.SEP_T_PWAM_FLAGS)
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    assert "backbone.layers.0.fusion.W_t.0.weight" in sd and tuple(sd["backbone.layers.0.fusion.W_t.0.weight"].shape[2:]) == (3, 3, 3)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=window, fusion_heads=mha, sep_t_pwam=True)
    x, l, m = O.synthetic_inputs(2, T, HW[0], HW[1], Nl=11)
    xv = x.permute(0, 2, 1, 3, 4)
    with torch.no_grad():
        ref = bb(xv, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, xv, l, m.unsqueeze(-1))
    for i, (a, b) in enumerate(zip(got, ref)):
        assert a.shape == b.shape
        err = (a - b).abs().max().item()
        assert err < 2e-4, f"stage {i}: max err {err}"
    # the oracle's random state dict carries the same keys / shapes as the reference module
    rsd = O.random_state_dict(cfg)
    for k, v in sd.items():
        if k.startswith("backbone.layers.0.fusion."):
            assert tuple(rsd[k].shape) == tuple(v.shape), k


@pytest.mark.parametrize("window,HW,mha", [(7, (64, 80), (1, 1, 1, 1)), (12, (96, 72), (1, 2, 2, 4)), (12, (40, 40), (1, 1, 1, 1))])
def test_image_backbone_matches_reference(window, HW, mha):
    """2-D twins (lib/backbone.py): never-clamped windows, per-call mask, (B,HW,C) token layout."""
    bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=window, mha=mha)
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, window, window), fusion_heads=mha, clamp_window=False, video=False)
    x, l, m = O.synthetic_inputs(2, 1, HW[0], HW[1], Nl=13, video=False)
    with torch.no_grad():
        ref = bb(x, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
        for i, (a, b) in enumerate(zip(got, ref)):
            assert a.shape == b.shape
            assert (a - b).abs().max().item() < 2e-4, f"stage {i}"
        assert (dec(ref[3], ref[2], ref[1], ref[0]) - O.decoder_forward(sd, got[3], got[2], got[1], got[0])).abs().max().item() < 2e-4


def test_random_state_dict_matches_reference_keys():
    net, _ = ref_shims.build_reference("lavt_video", "tiny")
    ref_sd = {k: v for k, v in net.state_dict().items() if not k.startswith("text_encoder.")}
    cfg = O.OracleConfig.swin("tiny")
    sd = O.random_state_dict(cfg)
    skip = ("relative_position_index", "num_batches_tracked")
    ref_keys = {k for k in ref_sd if not k.endswith(skip)}
    assert ref_keys == set(sd.keys())
    for k in ref_keys:
        assert tuple(ref_sd[k].shape) == tuple(sd[k].shape), k


def test_hs_backbone_matches_reference():
    """--hs: the stage outputs are the gated features (reference MMBasicLayer.forward :579-587)."""
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=(8, 7, 7), depths=(2, 2, 2, 2), extra=("--hs",))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(8, 7, 7), hs=True)
    x, l, m = O.synthetic_inputs(1, 4, 64, 64, Nl=11)
    xv = x.permute(0, 2, 1, 3, 4)
    with torch.no_grad():
        ref = bb(xv, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, xv, l, m.unsqueeze(-1))
    for i, (a, b) in enumerate(zip(got, ref)):
        assert (a - b).abs().max().item() < 2e-4, f"stage {i}"


@pytest.mark.parametrize("into_3d", [False, True])
def test_pretrained2d_inflation_matches_reference(tmp_path, into_3d):
    """LAVTVideo.load_from_pretrained2d_lavt_weights[_into_a_3d_model] (reference lib/_utils.py:133-238): same resulting
    state dict as the reference's own method, starting from a 2-D lavt_one checkpoint with window 12 -> video window (8,7,7)
    (bicubic resize of the bias tables + temporal tiling + patch-embed unsqueeze)."""
    ref2d, _ = ref_shims.build_reference("lavt_one", "tiny", window12=True, seed=3)
    ckpt = tmp_path / "lavt2d.pth"
    torch.save({"model": ref2d.state_dict()}, ckpt)
    ref3d, _ = ref_shims.build_reference("lavt_video", "tiny", seed=4)
    import contextlib
    import io
    name = "load_from_pretrained2d_lavt_weights_into_a_3d_model" if into_3d else "load_from_pretrained2d_lavt_weights"
    with contextlib.redirect_stdout(io.StringIO()):
        getattr(ref3d, name)(str(ckpt))
    from lavt_rs_b200.weights import inflate_lavt2d_state_dict
    before = {k: v.clone() for k, v in ref_shims.build_reference("lavt_video", "tiny", seed=4)[0].state_dict().items()}
    got = inflate_lavt2d_state_dict(ref2d.state_dict(), (8, 7, 7), before, drop_fusion=into_3d)
    want = ref3d.state_dict()
    checked = 0
    for k, v in got.items():
        if k not in want or want[k].shape != v.shape:
            continue                      # (2-D fusion keys that the video model does not have / cannot take)
        assert torch.equal(want[k], v) or torch.allclose(want[k], v, atol=1e-6), k
        checked += 1
    tables = [k for k in got if "relative_position_bias_table" in k]
    assert len(tables) == 12 and all(got[k].shape[0] == 15 * 13 * 13 for k in tables)
    assert got["backbone.patch_embed.proj.weight"].dim() == 5 and checked > 100
    assert into_3d == (not any(".fusion" in k for k in got))


@pytest.mark.parametrize("extra,cfg_kw", [((), {}), (("--version", "no_gate"), {"version": "no_gate"}), (("--version", "none"), {"version": "none"}),
                                          (("--hs",), {"hs": True})])
def test_training_gradients_match_reference_autograd(extra, cfg_kw):
    """The GRADIENT oracle (autograd through oracle/lavt_oracle.py with train-mode BatchNorm and the [0.9, 1.1]-weighted cross-entropy)
    pinned against autograd through the unmodified reference modules in train() mode: loss, d l_feats and every parameter gradient.
    This is what tests/test_backward_gpu.py holds the sm_100a backward kernels to."""
    import torch.nn.functional as F
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=(8, 7, 7), depths=(2, 2, 2, 2), extra=extra)
    _randomise_norms([bb, dec])
    g = torch.Generator().manual_seed(5)
    for layer in bb.layers:          # the reference zero-initialises the gates: give them signal
        if hasattr(layer, "res_gate"):
            for k in (0, 2):
                layer.res_gate[k].weight.data.copy_(torch.randn(layer.res_gate[k].weight.shape, generator=g) * layer.res_gate[k].weight.shape[0] ** -0.5)
    sd = {k: v.clone() for k, v in _sd(bb, dec).items()}
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(8, 7, 7), **cfg_kw)
    x, l, m = O.synthetic_inputs(2, 4, 64, 48, Nl=9)
    target = torch.randint(0, 2, (8, 64, 48), generator=g)
    bb.train()
    dec.train()
    lr_ = l.clone().requires_grad_()
    feats = bb(x.permute(0, 2, 1, 3, 4), lr_, m.unsqueeze(-1))
    out = F.interpolate(dec(feats[3], feats[2], feats[1], feats[0]), size=(64, 48), mode="bilinear", align_corners=True)
    loss_ref = F.cross_entropy(out, target, weight=torch.tensor([0.9, 1.1]))
    loss_ref.backward()
    ref = {"backbone." + k: p.grad for k, p in bb.named_parameters() if p.grad is not None}
    ref.update({"classifier." + k: p.grad for k, p in dec.named_parameters() if p.grad is not None})

    leaf = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in sd.items()}
    lo = l.clone().requires_grad_()
    loss = O.weighted_cross_entropy(O.model_forward(leaf, cfg, x, lo, m, train_bn=True), target)
    loss.backward()
    assert abs(loss.item() - loss_ref.item()) < 1e-5
    assert (lo.grad - lr_.grad).abs().max().item() < 1e-6 + 1e-3 * lr_.grad.abs().max().item()
    got = {k: v.grad for k, v in leaf.items() if v.grad is not None}
    assert set(got) == set(ref), set(got) ^ set(ref)
    for k, r in ref.items():
        err = (got[k] - r).norm().item() / (r.norm().item() + 1e-12)
        # fp32 on both sides; different op order (index-math gathers vs roll / partition copies) leaves ~1e-3 on the deepest tensors
        assert err < 5e-3 or (got[k] - r).abs().max().item() < 1e-7, (k, err)


def test_fuse_simple_matches_reference():
    """--fuse simple: PWAM with LangProject (mean-pooled sentence vector) instead of pixel-word attention (:916-917, 1012-1039)."""
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=(8, 7, 7), depths=(2, 2, 2, 2), extra=("--fuse", "simple"))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    assert "backbone.layers.0.fusion.image_lang_att.project.0.weight" in sd
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(8, 7, 7), fuse_simple=True)
    assert set(O.random_state_dict(cfg)) - {k for k in sd} == set()
    x, l, m = O.synthetic_inputs(2, 4, 64, 48, Nl=9)
    xv = x.permute(0, 2, 1, 3, 4)
    with torch.no_grad():
        ref = bb(xv, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, xv, l, m.unsqueeze(-1))
    for i, (a, b) in enumerate(zip(got, ref)):
        assert (a - b).abs().max().item() < 2e-4, i


def test_gacd_image_backbone_matches_reference():
    """--gacd: GA-CD fusion (lib/bcam.py:78-127) in the 2-D image backbone (lib/backbone.py:578-582)."""
    bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=7, depths=(2, 2, 2, 2), extra=("--gacd",))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    assert "backbone.layers.0.fusion.key_d.weight" in sd
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, 7, 7), clamp_window=False, video=False, gacd=True)
    assert {k for k in O.random_state_dict(cfg) if "fusion" in k} == {k for k in sd if "fusion" in k}
    x, l, m = O.synthetic_inputs(2, 1, 64, 80, Nl=11, video=False)
    with torch.no_grad():
        ref = bb(x, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
    for i, (a, b) in enumerate(zip(got, ref)):
        assert a.shape == b.shape and (a - b).abs().max().item() < 2e-4, i


def test_bcam_image_backbone_matches_reference():
    """--bcam: BCAM fusion (lib/bcam.py:8-75) in the 2-D image backbone; its Linear(dim -> hw) pins the input to 480 x 480."""
    bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=7, depths=(2, 2, 2, 2), extra=("--bcam",))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, 7, 7), clamp_window=False, video=False, bcam=True)
    assert {k for k in O.random_state_dict(cfg) if "fusion" in k} == {k for k in sd if "fusion" in k}
    x, l, m = O.synthetic_inputs(1, 1, 480, 480, Nl=9, video=False)
    with torch.no_grad():
        ref = bb(x, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
    for i, (a, b) in enumerate(zip(got, ref)):
        assert a.shape == b.shape and (a - b).abs().max().item() < 5e-4, (i, (a - b).abs().max().item())


def test_efn_image_backbone_matches_reference():
    """--efn: EFN fusion (lib/bcam.py:160-269) in the 2-D image backbone; 480 x 480 so that stages 0-2 pool (square maps of 120, 60, 30) and
    stage 3 (15 x 15 = 225 tokens) does not."""
    bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=7, depths=(2, 2, 2, 2), extra=("--efn",))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, 7, 7), clamp_window=False, video=False, efn=True)
    assert {k for k in O.random_state_dict(cfg) if "fusion" in k} == {k for k in sd if "fusion" in k}
    for k, v in O.random_state_dict(cfg).items():
        assert "fusion" not in k or v.shape == sd[k].shape, k
    x, l, m = O.synthetic_inputs(1, 1, 480, 480, Nl=9, video=False)
    with torch.no_grad():
        ref = bb(x, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
    # at random init the co-attention maps are almost uniform, so Lp / Mp barely vary over the tokens and the closing InstanceNorm
    # amplifies fp32 summation-order noise (the restatement contracts (B, n, C) rows, the reference (B, C, n) planes): 2e-3 on O(1) values
    for i, (a, b) in enumerate(zip(got, ref)):
        assert a.shape == b.shape and (a - b).abs().max().item() < 2e-3, (i, (a - b).abs().max().item())


def test_lazy_pred_model_matches_reference():
    """--lazy_pred (reference lib/video_swin_transformer.py:556-558, 586-587; lib/mask_predictor.py:32, 77; lib/_utils.py:101-107): stage
    outputs are the features BEFORE fusion at stages 1-3 and the decoder stops at 1/8 scale; whole video model without the text encoder."""
    import torch.nn.functional as F
    bb, dec, _ = ref_shims.build_reference_backbone_small(window=(8, 7, 7), depths=(2, 2, 2, 2), extra=("--lazy_pred",), out_indices=(1, 2, 3))
    _randomise_norms([bb, dec])
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(8, 7, 7), lazy_pred=True)
    mine = O.random_state_dict(cfg)
    benign = ("relative_position_index", "num_batches_tracked")          # buffers the oracle derives in closed form / does not need
    assert set(mine) == {k for k in sd if not k.endswith(benign)} and all(mine[k].shape == sd[k].shape for k in mine)
    x, l, m = O.synthetic_inputs(1, 4, 64, 64, Nl=11)
    xv = x.permute(0, 2, 1, 3, 4)
    with torch.no_grad():
        c2, c3, c4 = bb(xv, l, m.unsqueeze(-1))
        ref = F.interpolate(dec(c4, c3, c2, None), size=(64, 64), mode="bilinear", align_corners=True)
        feats = O.backbone_forward(sd, cfg, xv, l, m.unsqueeze(-1))
        got = O.model_forward(sd, cfg, x, l, m)
    assert len(feats) == 3
    for i, (a, b) in enumerate(zip(feats, (c2, c3, c4))):
        assert a.shape == b.shape and (a - b).abs().max().item() < 2e-4, f"stage {i + 1}"
    assert got.shape == ref.shape == (4, 2, 64, 64) and (got - ref).abs().max().item() < 2e-4


def test_vlt_head_matches_reference(monkeypatch):
    """oracle/vlt_oracle.py vs the unmodified reference VLTFuseAndClassify (lib/vlt.py:12-199) in eval mode, on CPU.  The reference's
    vlt_concat_coords builds its coordinate grids on the hard-coded device string 'cuda:<index>' (:268); only torch.arange's device
    argument is redirected here, the reference code itself runs untouched."""
    ref_shims.install_shims()
    from lib.vlt import VLTFuseAndClassify
    from oracle import vlt_oracle as VO
    real_arange = torch.arange

    def arange_on_cpu(*a, **kw):
        if isinstance(kw.get("device"), str) and kw["device"].startswith("cuda"):
            kw["device"] = "cpu"
        return real_arange(*a, **kw)
    monkeypatch.setattr(torch, "arange", arange_on_cpu)
    args = ref_shims.reference_args(["--model", "lavt_vlt", "--img_size", "128"])
    torch.manual_seed(0)
    head = VLTFuseAndClassify(d_model=256, nhead=8, d_hid=256, nlayers=2, args=args).eval()
    _randomise_norms([head])
    g = torch.Generator().manual_seed(7)
    for m in head.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.add_(0.1 * torch.randn(m.running_mean.shape, generator=g))
            m.running_var.add_(0.2 * torch.rand(m.running_var.shape, generator=g))
    sd = {k: v.detach() for k, v in head.state_dict().items()}
    B, Nl = 2, 11
    c4, c3, c2 = (torch.randn(B, 1024, 4, 4, generator=g), torch.randn(B, 512, 8, 8, generator=g), torch.randn(B, 256, 16, 16, generator=g))
    l = torch.randn(B, 768, Nl, generator=g)
    mask = torch.zeros(B, Nl, 1)
    mask[0, :8] = 1
    mask[1, :5] = 1
    with torch.no_grad():
        ref = head(c4, c3, c2, l, mask)
        got = VO.vlt_fuse_and_classify(sd, c4, c3, c2, l, mask)
    assert got.shape == ref.shape == (B, 2, 64, 64)
    assert (got - ref).abs().max().item() < 2e-4 * max(1.0, ref.abs().max().item()), (got - ref).abs().max().item()


@pytest.mark.parametrize("window,HW", [(7, (64, 80)), (12, (96, 72))])
def test_plain_swin_backbone_matches_reference(window, HW):
    """Plain Swin encoder of the ``vlt`` model (lib/backbone.py:1512-1650, no language fusion, out_indices (1, 2, 3)): the oracle's
    ``version='swin'`` mode vs the unmodified reference SwinTransformer."""
    ref_shims.install_shims()
    from lib.backbone import SwinTransformer
    torch.manual_seed(0)
    bb = SwinTransformer(embed_dim=128, depths=[2, 2, 2, 2], num_heads=[4, 8, 16, 32], window_size=window, ape=False, drop_path_rate=0.0,
                         patch_norm=True, out_indices=(1, 2, 3), use_checkpoint=False)
    bb.init_weights()
    bb.eval()
    _randomise_norms([bb])
    sd = {"backbone." + k: v.detach() for k, v in bb.state_dict().items()}
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, window, window), clamp_window=False, video=False, version="swin")
    x, l, m = O.synthetic_inputs(2, 1, HW[0], HW[1], Nl=5, video=False)
    with torch.no_grad():
        ref = bb(x)
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
    assert len(ref) == len(got) == 3
    for i, (a, b) in enumerate(zip(got, ref)):
        assert a.shape == b.shape
        assert (a - b).abs().max().item() < 2e-4, f"stage {i + 1}"


@pytest.mark.parametrize("extra,cfgkw", [(("--att_norm_layer_type", "BN"), dict(att_norm="BN")), (("--att_norm_layer_type", "LN"), dict(att_norm="LN")),
                                         (("--att_norm_layer_type", "none"), dict(att_norm="none")), (("--lg_act_layer", "sigmoid"), dict(gate_act="sigmoid")),
                                         (("--interpolate_before_seg",), dict(interpolate_before_seg=True)),
                                         (("--interpolate_before_seg", "--seg_last"), dict(interpolate_before_seg=True, seg_last=True))])
def test_image_backbone_flag_variants_match_reference(extra, cfgkw):
    """2-D backbone options --att_norm_layer_type BN | LN | none (lib/backbone.py:1297-1316), --lg_act_layer sigmoid (:552-554, :608) and the
    decoder levels of --interpolate_before_seg / --seg_last (lib/mask_predictor.py:40-48, 88-97): oracle vs the unmodified reference modules."""
    bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=7, extra=extra)
    _randomise_norms([bb, dec])
    g = torch.Generator().manual_seed(3)
    for m in bb.modules():
        if isinstance(m, torch.nn.BatchNorm1d):
            m.running_mean.add_(0.1 * torch.randn(m.running_mean.shape, generator=g))
            m.running_var.add_(0.2 * torch.rand(m.running_var.shape, generator=g))
    sd = _sd(bb, dec)
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(1, 7, 7), clamp_window=False, video=False, **cfgkw)
    x, l, m = O.synthetic_inputs(2, 1, 64, 80, Nl=13, video=False)
    with torch.no_grad():
        ref = bb(x, l, m.unsqueeze(-1))
        got = O.backbone_forward(sd, cfg, x, l, m.unsqueeze(-1))
        for i, (a, b) in enumerate(zip(got, ref)):
            assert (a - b).abs().max().item() < 2e-4, f"stage {i}"
        rl = dec(ref[3], ref[2], ref[1], ref[0])
        gl = O.decoder_forward(sd, got[3], got[2], got[1], got[0])
        assert rl.shape == gl.shape and (rl - gl).abs().max().item() < 2e-4
    # the oracle's random state dict carries the variant's extra keys with the reference's shapes
    rsd = O.random_state_dict(cfg)
    assert {k: tuple(v.shape) for k, v in rsd.items()} == {k: tuple(v.shape) for k, v in sd.items()
                                                           if not k.endswith(("relative_position_index", "num_batches_tracked"))}


def test_losses_match_reference():
    """lavt_rs_b200/losses.py vs the reference's losses.py (:38-243): value and gradient w.r.t. the logits for every --loss option."""
    ref_shims.install_shims()
    import importlib
    ref_losses = importlib.import_module("losses")
    from lavt_rs_b200 import losses as mine
    g = torch.Generator().manual_seed(11)
    logits = torch.randn(3, 2, 24, 20, generator=g)
    target = (torch.rand(3, 24, 20, generator=g) > 0.6).long()
    target[:, 5:15, 4:12] = 1
    pairs = [(ref_losses.MultiClassDiceLoss(), mine.MultiClassDiceLoss()), (ref_losses.DiceFocalLoss(3, 1), mine.DiceFocalLoss(3, 1)),
             (ref_losses.DiceBoundaryLoss(0.05, 1), mine.DiceBoundaryLoss(0.05, 1)), (ref_losses.DiceFocalLoss(0.5, 2.0), mine.DiceFocalLoss(0.5, 2.0))]
    for r, m in pairs:
        a = logits.clone().requires_grad_()
        b = logits.clone().requires_grad_()
        lr, lm = r(a, target), m(b, target)
        lr.backward()
        lm.backward()
        assert abs(lr.item() - lm.item()) < 1e-6 * max(1.0, abs(lr.item())), type(m).__name__
        assert (a.grad - b.grad).abs().max().item() < 1e-7 + 1e-5 * a.grad.abs().max().item(), type(m).__name__
    bl_r, bl_m = ref_losses.BoundaryLoss(), mine.BoundaryLoss()
    prob, hot = logits.softmax(1), mine.one_hot(target, 2, dtype=torch.float32)
    assert abs(bl_r(prob.clone(), hot.clone()).item() - bl_m(prob, hot).item()) < 1e-6
    assert torch.equal(ref_losses.one_hot(target, 2, dtype=torch.float32), hot)
    ce = torch.nn.functional.cross_entropy(logits, target, weight=torch.tensor([0.9, 1.1]))      # the reference's version calls .cuda()
    assert abs(mine.cross_entropy_loss(logits, target).item() - ce.item()) < 1e-7
    from lavt_rs_b200.args import default_args
    assert isinstance(mine.build_criterion(default_args(["--loss", "dice_boundary"])), mine.DiceBoundaryLoss)
    assert mine.build_criterion(default_args([])) is mine.cross_entropy_loss


def test_swin2d_inflation_matches_reference(tmp_path):
    """MultiModalSwinTransformer3D.inflate_weights (lib/video_swin_transformer.py:759-805): ImageNet 2-D Swin checkpoint -> video backbone,
    this repo's method vs the unmodified reference method on the same synthetic checkpoint (window 7 tables into an 8 x 12 x 12 model)."""
    import contextlib
    import io
    from lavt_rs_b200.lib.video_swin_transformer import MultiModalSwinTransformer3D as Mine
    bb, _, _ = ref_shims.build_reference_backbone_small(window=(8, 12, 12))
    g = torch.Generator().manual_seed(2)
    sd2d = {}
    for k, v in bb.state_dict().items():
        if "fusion" in k or "res_gate" in k or k.startswith("norm"):
            continue
        if "relative_position_bias_table" in k:
            sd2d[k] = torch.randn(13 * 13, v.shape[1], generator=g)
        elif k == "patch_embed.proj.weight":
            sd2d[k] = torch.randn(v.shape[0], 3, 4, 4, generator=g)
        elif "relative_position_index" in k:
            sd2d[k] = torch.zeros(49, 49, dtype=torch.long)
        else:
            sd2d[k] = torch.randn(v.shape, generator=g)
    path = str(tmp_path / "swin2d.pth")
    torch.save({"model": sd2d}, path)
    mine = Mine(patch_size=(1, 4, 4), embed_dim=128, depths=[2, 2, 2, 2], num_heads=[4, 8, 16, 32], window_size=(8, 12, 12), drop_path_rate=0.0,
                patch_norm=True, args=None)
    bb.pretrained, mine.pretrained = path, path
    with contextlib.redirect_stdout(io.StringIO()):
        bb.inflate_weights()
        mine.inflate_weights()
    rs, ms = bb.state_dict(), mine.state_dict()
    for k in sd2d:
        if "relative_position_index" in k:
            continue
        assert torch.equal(rs[k], ms[k]), k
    assert ms["layers.0.blocks.0.attn.relative_position_bias_table"].shape == (15 * 23 * 23, 4)
