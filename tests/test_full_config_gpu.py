"""BASELINE.json configs[1] / configs[2] at their REAL size on the CUDA path: Video Swin-B (depths 2-2-18-2, embed 128, heads 4-8-16-32),
one clip of 8 x 384 x 384 frames, 20-word expression, window (8,7,7) and --window12 (8,12,12) -- reference builder
lib/segmentation.py:154-211.

Checked against BOTH
  * the CPU oracle run here on the same seeded weights / inputs: every stage output c1..c4 and the logits in full, and
  * the golden file written by the UNMODIFIED reference (oracle/make_golden.py full_* cases: strided slices of every tensor, whole-tensor
    norms, the reference's thresholded mask bit for bit and its fp32 logit margin quantised to int8, both at every second pixel).

Tolerances (north_star): per-layer outputs and logits within 2e-2 (rel-L2; bf16 operands, fp32 accumulation); thresholded masks agree
on >= 99.9 % of the pixels whose fp32 margin is resolvable.  With random-init weights the two logits of a pixel differ by ~0.03 (std)
while a bf16 forward moves a logit by ~3e-4, so ~2.5 % of ALL pixels sit within one error bar of the decision boundary: the raw
all-pixel agreement is reported and bounded by what that density predicts, the 99.9 % bar is asserted on pixels whose reference margin
exceeds 4x the measured max logit error (the same filter for both windows)."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import lavt_oracle as O  # noqa: E402  (checker)
from oracle.make_golden import CASES, OUT, case_inputs, subsample, subsample_mask  # noqa: E402

pytestmark = pytest.mark.gpu

TOL = 2e-2


def rel_l2(a, b):
    a, b = a.float().cpu(), torch.as_tensor(np.asarray(b)).float()
    return ((a - b).norm() / (b.norm() + 1e-12)).item()


def _build(c):
    from lavt_rs_b200.lib._utils import LAVT
    from lavt_rs_b200.lib.mask_predictor import SimpleDecoding
    from lavt_rs_b200.lib.video_swin_transformer import MultiModalSwinTransformer3D
    from lavt_rs_b200.weights import load_reference_state_dict
    cfg, sd, x, l, m = case_inputs(c)
    bb = MultiModalSwinTransformer3D(patch_size=(1, 4, 4), embed_dim=128, depths=list(c["depths"]), num_heads=[4, 8, 16, 32],
                                     window_size=c["window"], drop_path_rate=0.0, patch_norm=True, num_heads_fusion=list(c["mha"]), args=None)
    dec = SimpleDecoding(1024, None)
    load_reference_state_dict(bb, sd, "backbone.")
    load_reference_state_dict(dec, sd, "classifier.")
    return cfg, sd, x, l, m, bb, dec, LAVT(bb, dec).cuda().eval()


@pytest.mark.parametrize("name", ["full_w7_t8_384", "full_w12_t8_384"])
def test_baseline_video_config_full_depth(name):
    c = CASES[name]
    gold = np.load(os.path.join(OUT, name + ".npz"))
    cfg, sd, x, l, m, bb, dec, model = _build(c)
    with torch.no_grad():
        feats = bb(x.permute(0, 2, 1, 3, 4).cuda(), l.cuda(), m.unsqueeze(-1).cuda())
        logits = model._segment(x.cuda().permute(0, 2, 1, 3, 4), l.cuda(), m.cuda(), (c["H"], c["W"])).float().cpu()
        cap = {}
        ref_logits = O.model_forward(sd, cfg, x, l, m, capture=cap)        # CPU oracle, same seeds
    report = {}
    # ---- per-stage outputs and logits: full tensors vs the oracle, strided slices + norms vs the reference's golden file
    for i in range(4):
        key = f"c{i + 1}"
        assert feats[i].shape == cap[key].shape
        report[key] = (rel_l2(feats[i], cap[key]), rel_l2(subsample(key, feats[i]), gold[key]))
        assert report[key][0] < TOL, f"{name}: stage output {key} rel-L2 vs oracle {report[key][0]:.3e}"
        assert report[key][1] < TOL, f"{name}: stage output {key} rel-L2 vs reference golden slice {report[key][1]:.3e}"
        assert abs(feats[i].float().norm().item() / float(gold[key + "_norm"]) - 1) < 5e-3, key
    report["logits"] = (rel_l2(logits, ref_logits), rel_l2(subsample("logits", logits), gold["logits"]))
    assert report["logits"][0] < TOL and report["logits"][1] < TOL, f"{name}: logits rel-L2 {report['logits']}"
    # ---- thresholded masks vs the REFERENCE's mask (golden, bit-packed) and vs the oracle's
    ours = subsample_mask(logits[:, 1] > logits[:, 0]).numpy()                               # the stored pixels (MASK_STRIDE)
    ref_mask = np.unpackbits(gold["mask_bits"])[: ours.size].reshape(ours.shape).astype(bool)
    assert (subsample_mask(ref_logits[:, 1] > ref_logits[:, 0]).numpy() == ref_mask).mean() > 0.9999   # oracle == reference (fp32 ties)
    margin = np.abs(gold["margin_q"].astype(np.float32)) * float(gold["margin_step"])         # reference's |logit_1 - logit_0|
    err = (logits - ref_logits).abs().max().item()
    agree_all = float((ours == ref_mask).mean())
    clear = margin > 4 * err + float(gold["margin_step"])
    agree_clear = float((ours == ref_mask)[clear].mean())
    # expected raw disagreement if the error were uniform: P(|margin| < |err_pixel|); bounded by the fraction of pixels within max err
    near = float((margin <= err).mean())
    report["mask"] = dict(all=agree_all, clear=agree_clear, clear_fraction=float(clear.mean()), max_logit_err=err, within_err=near)
    print(name, report)
    assert clear.mean() > 0.5, "the margin filter must keep most pixels"
    assert agree_clear >= 0.999, f"{name}: mask agreement on resolvable pixels {agree_clear:.5f}"
    assert 1.0 - agree_all <= near + 1e-4, f"{name}: {1 - agree_all:.4%} of all pixels flip but only {near:.4%} lie within the logit error"
    assert agree_all >= 0.99, f"{name}: raw mask agreement {agree_all:.5f}"
