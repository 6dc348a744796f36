"""Generate tests/golden/*.npz from the UNMODIFIED reference (needs the reference checkout, see oracle/ref_shims.py).

    python oracle/make_golden.py [case ...]

For each case: seeded weights (oracle.random_state_dict -- deterministic torch.Generator streams) are loaded
INTO the reference's own nn.Modules (MultiModalSwinTransformer3D + SimpleDecoding, imported from its checkout
through oracle/ref_shims.py), the reference forward is executed on seeded synthetic inputs, and its outputs are
stored.  tests/test_oracle_golden.py replays the same seeds through the oracle (CPU) and, on the GPU box,
tests/test_golden_gpu.py through the CUDA path -- the reference itself never travels.
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

CASES = {
    # name: (window, depths, fusion heads, B, T, H, W, Nl, stored stage outputs)
    "w7_t4_32": dict(window=(8, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=1, T=4, H=32, W=32, Nl=20, keep=(0, 1, 2, 3)),
    "w12_t2_48": dict(window=(8, 12, 12), depths=(2, 2, 2, 2), mha=(1, 2, 4, 8), B=2, T=2, H=48, W=48, Nl=9, keep=(1, 2, 3)),
    "w7_t16_32x40": dict(window=(8, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=1, T=16, H=32, W=40, Nl=22, keep=(2, 3)),
    # README video configuration: SepTPWAM fusion (--sep_t_pwam --conv3d_kernel_size_t 3-3-3 --conv3d_kernel_size_s 1-1-1
    # --w_t3x3_s1x1 --mm_t3x3_s1x1)
    "sept_w7_t4_32": dict(window=(8, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 2, 2), B=1, T=4, H=32, W=32, Nl=20, keep=(0, 1, 2, 3),
                          sep_t_pwam=True),
    # 2-D image backbone (lib/backbone.py): window is an int, never clamped
    "img_w12_60x76": dict(window=(1, 12, 12), depths=(2, 2, 2, 2), mha=(1, 1, 2, 2), B=2, T=1, H=60, W=76, Nl=20, keep=(1, 2, 3),
                          image=True),
    # fusion ablations of lib/bcam.py in the 2-D image backbone (flags = the reference's own CLI flags) and --lazy_pred
    "img_efn_128": dict(window=(1, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=1, T=1, H=128, W=128, Nl=20, keep=(1, 2, 3), image=True,
                        flags=("--efn",)),                      # 32 x 32 and 16 x 16 maps are pooled (hw > 225), 8 x 8 and 4 x 4 are not
    "img_gacd_64x96": dict(window=(1, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=2, T=1, H=64, W=96, Nl=20, keep=(1, 2, 3), image=True,
                           flags=("--gacd",)),
    "img_bcam_480": dict(window=(1, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=1, T=1, H=480, W=480, Nl=20, keep=(), image=True,
                         flags=("--bcam",), store_logits=False),   # a_proj pins BCAM to 480 x 480; only the 1/4-scale logits are stored
    "lazy_w7_t4_64": dict(window=(8, 7, 7), depths=(2, 2, 2, 2), mha=(1, 1, 1, 1), B=1, T=4, H=64, W=64, Nl=20, keep=(1, 2, 3),
                          flags=("--lazy_pred",)),
    # BASELINE.json configs[1] / configs[2] at their REAL size: Video Swin-B depths 2-2-18-2, one clip of 8 x 384 x 384, 20 words, window
    # (8,7,7) and --window12.  The full tensors are 60 MB, so strided slices (``subsample`` below) + per-tensor statistics are stored.
    "full_w7_t8_384": dict(window=(8, 7, 7), depths=(2, 2, 18, 2), mha=(1, 1, 1, 1), B=1, T=8, H=384, W=384, Nl=20, keep=(0, 1, 2, 3),
                           sub=True),
    "full_w12_t8_384": dict(window=(8, 12, 12), depths=(2, 2, 18, 2), mha=(1, 1, 1, 1), B=1, T=8, H=384, W=384, Nl=20, keep=(0, 1, 2, 3),
                            sub=True),
}
OUT = os.path.join(ROOT, "tests", "golden")

# strided slices stored for the full-size cases: (channel stride, spatial stride) per tensor
SUB = {"c1": (32, 4), "c2": (64, 2), "c3": (64, 1), "c4": (32, 1), "logits": (1, 8), "logits_lowres": (1, 2)}
MASK_STRIDE = 2     # pixel stride of the stored mask and margin maps (keeps each file under 1 MB)


def subsample(key: str, t):
    """The slice of tensor ``key`` ([frames, C, H, W]) that a ``sub=True`` golden case stores."""
    cs, ss = SUB[key]
    return t[:, ::cs, ::ss, ::ss]


def subsample_mask(t):
    """The pixels ([frames, H, W]) of the mask and margin maps that a ``sub=True`` golden case stores."""
    return t[:, ::MASK_STRIDE, ::MASK_STRIDE]


def case_inputs(c):
    image = c.get("image", False)
    cfg = O.OracleConfig(depths=c["depths"], window=c["window"], fusion_heads=c["mha"], clamp_window=not image, video=not image,
                         sep_t_pwam=c.get("sep_t_pwam", False), **{f[2:]: True for f in c.get("flags", ())})
    sd = O.random_state_dict(cfg, seed=0)
    x, l, m = O.synthetic_inputs(c["B"], c["T"], c["H"], c["W"], Nl=c["Nl"], seed=1, video=not image)
    return cfg, sd, x, l, m


def main():
    os.makedirs(OUT, exist_ok=True)
    only = set(sys.argv[1:])
    for name, c in CASES.items():
        if only and name not in only:
            continue
        cfg, sd, x, l, m = case_inputs(c)
        flags = tuple(c.get("flags", ()))
        lazy = "--lazy_pred" in flags
        if c.get("image", False):
            bb, dec, _ = ref_shims.build_reference_image_backbone_small(window=c["window"][1], mha=c["mha"], depths=c["depths"], extra=flags)
        else:
            bb, dec, _ = ref_shims.build_reference_backbone_small(window=c["window"], mha=c["mha"], depths=c["depths"],
                                                                  extra=(ref_shims.SEP_T_PWAM_FLAGS if c.get("sep_t_pwam") else ()) + flags,
                                                                  out_indices=(1, 2, 3) if lazy else (0, 1, 2, 3))
        missing = bb.load_state_dict({k[len("backbone."):]: v for k, v in sd.items() if k.startswith("backbone.")}, strict=False)
        assert all(k.endswith("relative_position_index") for k in missing.missing_keys) and not missing.unexpected_keys, missing
        missing = dec.load_state_dict({k[len("classifier."):]: v for k, v in sd.items() if k.startswith("classifier.")}, strict=False)
        assert all(k.endswith("num_batches_tracked") for k in missing.missing_keys) and not missing.unexpected_keys, missing
        with torch.no_grad():
            feats = bb(x if c.get("image", False) else x.permute(0, 2, 1, 3, 4), l, m.unsqueeze(-1))   # reference forward
            feats = ((None,) + tuple(feats)) if lazy else tuple(feats)                                   # lib/_utils.py:101-105
            low = dec(feats[3], feats[2], feats[1], feats[0])
            logits = F.interpolate(low, size=(c["H"], c["W"]), mode="bilinear", align_corners=True)   # lib/_utils.py:106
        sub = (lambda k, t: subsample(k, t)) if c.get("sub") else (lambda k, t: t)
        arrays = {"logits_lowres": sub("logits_lowres", low).numpy()}
        if c.get("store_logits", True):
            arrays["logits"] = sub("logits", logits).numpy()
        for i in c["keep"]:
            arrays[f"c{i + 1}"] = sub(f"c{i + 1}", feats[i]).numpy()
        if c.get("sub"):
            # whole-tensor statistics of what was not stored: L2 norm of every tensor, the thresholded mask (bit-packed) and the
            # fp32 logit margin quantised to int8 are what the mask-agreement checks need
            arrays["logits_norm"] = np.float32(logits.norm().item())
            arrays["mask_bits"] = np.packbits(subsample_mask(logits[:, 1] > logits[:, 0]).numpy())
            margin = (logits[:, 1] - logits[:, 0]).numpy()
            step = float(margin.std()) / 32.0                      # int8 steps of std/32: fine where it matters (around zero)
            arrays["margin_step"] = np.float32(step)
            arrays["margin_q"] = np.clip(np.rint(subsample_mask(margin) / step), -127, 127).astype(np.int8)
            for i in range(4):
                arrays[f"c{i + 1}_norm"] = np.float32(feats[i].norm().item())
        for i in range(4):
            if feats[i] is not None:
                arrays[f"c{i + 1}_absmean"] = np.float32(feats[i].abs().mean().item())
        path = os.path.join(OUT, name + ".npz")
        np.savez_compressed(path, **arrays)
        print(name, {k: getattr(v, "shape", v) for k, v in arrays.items()}, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
