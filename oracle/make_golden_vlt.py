"""Golden outputs of the UNMODIFIED reference VLT head (lib/vlt.py: VLTFuseAndClassify) -> tests/golden/vlt_*.npz.

    python oracle/make_golden_vlt.py            (imports the reference checkout through oracle/ref_shims.py)

Weights: a seeded state dict built with this repo's parameter container (same names / shapes as the reference's module, checked by
load_state_dict(strict=True) into the reference head), norms and BatchNorm statistics randomised so that every affine / running
statistic matters.  The reference's vlt_concat_coords hard-codes the device string 'cuda:<index>' (lib/vlt.py:268); as in
tests/test_oracle_vs_reference.py only torch.arange's device argument is redirected, the reference code itself runs untouched.
tests/test_oracle_golden.py replays the cases through oracle/vlt_oracle.py (CPU), tests/test_vlt_gpu.py through the CUDA path.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OUT = os.path.join(ROOT, "tests", "golden")
VLT_CASES = {
    # name: img_size (s = img_size / 16), batch, words, valid words per image
    "vlt_head_160": dict(img_size=160, B=2, Nl=11, valid=(8, 5)),
    "vlt_head_480": dict(img_size=480, B=1, Nl=20, valid=(14,)),      # the size the reference's README trains lavt_vlt at
}


def vlt_case(c):
    """(args, state dict, (c4, c3, c2, l, mask[B,Nl,1])) of a case: seeded, reproducible wherever the repo is."""
    from lavt_rs_b200.args import default_args
    from lavt_rs_b200.lib.vlt import VLTFuseAndClassify
    args = default_args(["--model", "lavt_vlt", "--img_size", str(c["img_size"])])
    torch.manual_seed(1234)
    head = VLTFuseAndClassify(d_model=256, nhead=8, d_hid=256, nlayers=2, args=args)
    g = torch.Generator().manual_seed(77)
    with torch.no_grad():
        for m in head.modules():
            if isinstance(m, (torch.nn.BatchNorm1d, torch.nn.BatchNorm2d)):
                m.weight.copy_(1.0 + 0.2 * torch.randn(m.weight.shape, generator=g))
                m.bias.copy_(0.1 * torch.randn(m.bias.shape, generator=g))
                m.running_mean.copy_(0.1 * torch.randn(m.running_mean.shape, generator=g))
                m.running_var.copy_(1.0 + 0.3 * torch.rand(m.running_var.shape, generator=g))
            elif isinstance(m, torch.nn.LayerNorm):
                m.weight.copy_(1.0 + 0.2 * torch.randn(m.weight.shape, generator=g))
                m.bias.copy_(0.1 * torch.randn(m.bias.shape, generator=g))
    sd = {k: v.detach().clone() for k, v in head.state_dict().items()}
    s, B, Nl = c["img_size"] // 16, c["B"], c["Nl"]
    c4 = torch.randn(B, 1024, s // 2, s // 2, generator=g)
    c3 = torch.randn(B, 512, s, s, generator=g)
    c2 = torch.randn(B, 256, 2 * s, 2 * s, generator=g)
    l = torch.randn(B, 768, Nl, generator=g)
    mask = torch.zeros(B, Nl, 1)
    for b, n in enumerate(c["valid"]):
        mask[b, :n] = 1
    return args, sd, (c4, c3, c2, l, mask)


def main():
    from oracle import ref_shims
    ref_shims.install_shims()
    from lib.vlt import VLTFuseAndClassify as RefHead
    real_arange = torch.arange

    def arange_on_cpu(*a, **kw):
        if isinstance(kw.get("device"), str) and kw["device"].startswith("cuda"):
            kw["device"] = "cpu"
        return real_arange(*a, **kw)
    torch.arange = arange_on_cpu
    try:
        for name, c in VLT_CASES.items():
            _, sd, (c4, c3, c2, l, mask) = vlt_case(c)
            rargs = ref_shims.reference_args(["--model", "lavt_vlt", "--img_size", str(c["img_size"])])
            ref = RefHead(d_model=256, nhead=8, d_hid=256, nlayers=2, args=rargs).eval()
            ref.load_state_dict(sd, strict=True)                      # same names, same shapes
            with torch.no_grad():
                out = ref(c4, c3, c2, l, mask)
            path = os.path.join(OUT, name + ".npz")
            np.savez_compressed(path, logits=out.numpy())
            print(name, tuple(out.shape), os.path.getsize(path) // 1024, "KiB")
    finally:
        torch.arange = real_arange


if __name__ == "__main__":
    main()
