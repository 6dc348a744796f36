"""Generate tests/golden/train_*.npz from the UNMODIFIED reference in train() mode (needs the reference checkout, see oracle/ref_shims.py).

    python oracle/make_golden_train.py

Seeded weights (oracle.random_state_dict, with non-zero LanguageGate weights) are loaded into the reference's own modules
(oracle/ref_shims.py), one training step is executed -- forward with batch-statistics BatchNorm, bilinear upsample, the
[0.9, 1.1]-weighted cross-entropy of losses.py:7-11, ``loss.backward()`` -- and the loss, the gradient of the language features, the
L2 norm of EVERY parameter gradient and a few gradient tensors (see ROWS) are stored.  tests/test_oracle_golden.py replays the seeds
through autograd of the oracle (CPU) and tests/test_golden_gpu.py through the sm_100a backward kernels.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import lavt_oracle as O  # noqa: E402
from oracle import ref_shims  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
TRAIN_CASES = {
    "train_w7_t4_64x48": dict(window=(8, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=2, T=4, H=64, W=48, Nl=11),
}
FULL = ("backbone.layers.0.blocks.1.attn.relative_position_bias_table", "backbone.layers.2.blocks.0.attn.qkv.bias",
        "backbone.layers.1.fusion.image_lang_att.f_key.0.weight", "backbone.layers.3.blocks.1.mlp.fc2.bias", "backbone.norm2.weight",
        "backbone.layers.0.downsample.norm.bias", "backbone.layers.1.res_gate.2.weight", "classifier.bn1_3.weight", "classifier.conv1_1.weight",
        "backbone.patch_embed.proj.weight")
ROWS = {"backbone.layers.1.fusion.image_lang_att.f_key.0.weight": 64}     # leading output channels stored (keeps the file under 1 MB)


def train_case_inputs(c):
    cfg = O.OracleConfig(depths=c["depths"], window=c["window"], fusion_heads=c["mha"])
    sd = O.random_state_dict(cfg, seed=0)
    g = torch.Generator().manual_seed(7)
    for s in range(4):      # the reference zero-initialises the gates: give them signal so that their path carries gradient
        C = cfg.embed_dim * 2 ** s
        for k in ("0", "2"):
            sd[f"backbone.layers.{s}.res_gate.{k}.weight"] = torch.randn(C, C, generator=g) * C ** -0.5
    x, l, m = O.synthetic_inputs(c["B"], c["T"], c["H"], c["W"], Nl=c["Nl"], seed=1)
    target = torch.randint(0, 2, (c["B"] * c["T"], c["H"], c["W"]), generator=g)
    return cfg, sd, x, l, m, target


def main():
    for name, c in TRAIN_CASES.items():
        cfg, sd, x, l, m, target = train_case_inputs(c)
        bb, dec, _ = ref_shims.build_reference_backbone_small(window=c["window"], mha=c["mha"], depths=c["depths"])
        bb.load_state_dict({k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}, strict=False)
        dec.load_state_dict({k[len("classifier."):]: v for k, v in sd.items() if k.startswith("classifier.")}, strict=False)
        bb.train()
        dec.train()
        lr = l.clone().requires_grad_()
        feats = bb(x.permute(0, 2, 1, 3, 4), lr, m.unsqueeze(-1))
        out = F.interpolate(dec(feats[3], feats[2], feats[1], feats[0]), size=(c["H"], c["W"]), mode="bilinear", align_corners=True)
        loss = F.cross_entropy(out, target, weight=torch.tensor([0.9, 1.1]))        # losses.py:7-11
        loss.backward()
        grads = {"backbone." + k: p.grad for k, p in bb.named_parameters() if p.grad is not None}
        grads.update({"classifier." + k: p.grad for k, p in dec.named_parameters() if p.grad is not None})
        names = sorted(grads)
        arrays = {"loss": np.float32(loss.item()), "dl": lr.grad.numpy(), "names": np.array(names),
                  "norms": np.array([grads[k].norm().item() for k in names], dtype=np.float32),
                  "bn1_4_running_mean": dec.bn1_4.running_mean.numpy()}
        for k in FULL:
            arrays["g:" + k] = grads[k][:ROWS.get(k)].numpy()
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(name, "loss", loss.item(), len(names), "gradients", os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
