"""The inference decoder's first conv of each level runs on the coarse grid: Z = W_tap . Y (GEMM), the skip half of the conv, and
upconv_blend, which assembles conv3x3(bilinear_up(Y)) from Z.  The blend is checked against torch fp32 from the same bf16 Z and fp32
skip part, the whole level against an fp32 conv over cat[interpolate(Y), skip], and the decoder against the CPU oracle."""
import os
import sys
import types

import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import lavt_oracle as O  # noqa: E402  (test infrastructure)

pytestmark = pytest.mark.gpu

SIZES = [((12, 12), (24, 24)), ((5, 6), (10, 11)), ((1, 1), (3, 3)), ((2, 3), (2, 3)), ((3, 2), (7, 5)),
         ((1, 3), (2, 6)), ((3, 2), (6, 4))]          # the last two: x2 maps of side 1 and 2


def _level(cy, cs, hid, seed):
    g = torch.Generator().manual_seed(seed)
    conv = torch.nn.Conv2d(cy + cs, hid, 3, padding=1, bias=False)
    conv.weight.data = torch.randn(hid, cy + cs, 3, 3, generator=g) / (3 * (cy + cs) ** 0.5)
    bn = torch.nn.BatchNorm2d(hid)
    bn.weight.data = torch.rand(hid, generator=g) + 0.5
    bn.bias.data = torch.rand(hid, generator=g) - 0.5
    bn.running_mean = torch.rand(hid, generator=g) * 0.4 - 0.2
    bn.running_var = torch.rand(hid, generator=g) + 0.5
    dec = types.SimpleNamespace(conv=conv.cuda().eval(), bn=bn.cuda().eval())
    from lavt_rs_b200 import engine as E
    dec.prepared = E.PreparedWeights()
    return dec


def _blend_ref(z, h, w, H, W, hid):
    """sum_tap shift_tap(interpolate(Z_tap)) in fp32, zero padding on the fine grid: conv3x3(up(Y)) with Z = W_tap . Y."""
    n = z.shape[0]
    zt = z.float().view(n, h, w, 9, hid).permute(0, 3, 4, 1, 2).reshape(n, 9 * hid, h, w)
    up = F.interpolate(zt, size=(H, W), mode="bilinear", align_corners=True).view(n, 9, hid, H, W)
    up = F.pad(up, (1, 1, 1, 1))
    acc = torch.zeros(n, hid, H, W, device=z.device)
    for ky in range(3):
        for kx in range(3):
            acc += up[:, ky * 3 + kx, :, ky:ky + H, kx:kx + W]
    return acc.permute(0, 2, 3, 1)


@pytest.mark.parametrize("hid", [384, 512])
@pytest.mark.parametrize("cs", [0, 96, 128])
@pytest.mark.parametrize("hw,HW", SIZES)
def test_upconv_level(hw, HW, cs, hid):
    from lavt_rs_b200 import engine as E
    (h, w), (H, W) = hw, HW
    n, cy = 2, 256
    dec = _level(cy, cs, hid, seed=h * 100 + W * 10 + cs + hid)
    g = torch.Generator().manual_seed(7)
    y = torch.randn(n, h, w, cy, generator=g).to(torch.bfloat16).cuda()
    skip = torch.randn(n, H, W, cs, generator=g).to(torch.bfloat16).cuda() if cs else None
    ws = E.Workspace()
    out = torch.empty(n, H, W, hid, device="cuda", dtype=torch.bfloat16)
    E._upconv_bn_relu(y, skip, dec, "conv", "bn", ws, out)
    torch.cuda.synchronize()
    s, b = E._bn_fold(dec.bn)

    # blend alone, at fp32 level from the same bf16 Z and fp32 skip part (the output is bf16: one rounding)
    z = ws.get("dec_z", (n, h, w, 9 * hid), torch.bfloat16, y.device)
    add = ws.get("dec_p", (n, H, W, hid), torch.float32, y.device) if cs else b
    ref = torch.relu(add + s * _blend_ref(z, h, w, H, W, hid))
    err = (out.float() - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 1e-5 * ref.pow(2).mean().sqrt()
    assert (err <= tol).all(), f"blend: max err {err.max().item():.3e}, worst excess {(err - tol).max().item():.3e}"

    # the whole level against conv3x3 + BN + ReLU of cat[interpolate(Y), skip] in fp32
    x = F.interpolate(y.float().permute(0, 3, 1, 2), size=(H, W), mode="bilinear", align_corners=True)
    if cs:
        x = torch.cat([x, skip.float().permute(0, 3, 1, 2)], 1)
    full = torch.relu(F.conv2d(x, dec.conv.weight.float(), padding=1) * s.view(1, -1, 1, 1) + b.view(1, -1, 1, 1)).permute(0, 2, 3, 1)
    rel = ((out.float() - full).norm() / full.norm()).item()
    assert rel < 1e-2, f"level rel-L2 {rel:.3e}"


@pytest.fixture(scope="module")
def decoder():
    from lavt_rs_b200.lib.mask_predictor import SimpleDecoding
    from lavt_rs_b200.weights import load_reference_state_dict
    cfg = O.OracleConfig(depths=(2, 2, 2, 2), window=(8, 7, 7))
    sd = O.random_state_dict(cfg, seed=0)
    dec = SimpleDecoding(1024, None)
    load_reference_state_dict(dec, sd, "classifier.")
    return sd, dec.cuda().eval()


def _feats(n, side, seed):
    g = torch.Generator().manual_seed(seed)
    return tuple(torch.randn(n, 128 * 2 ** i, side // 2 ** i, side // 2 ** i, generator=g) for i in range(4))


def test_decoder_x2_levels_match_oracle(decoder):
    """Every level an exact x2 upsample (the bench geometry, smaller), so the shared-memory blend kernel runs at all three."""
    sd, dec = decoder
    c1, c2, c3, c4 = _feats(3, 32, seed=5)
    ref = O.decoder_forward(sd, c4, c3, c2, c1)
    got = dec(c4.cuda(), c3.cuda(), c2.cuda(), c1.cuda())
    a, r = got.float().cpu(), ref.float()
    rms = r.pow(2).mean().sqrt().item()
    bad = ((a - r).abs() > 2e-2 * r.abs() + 2e-2 * rms).float().mean().item()
    rel = ((a - r).norm() / r.norm()).item()
    assert bad < 1e-4 and rel < 1e-2, f"decoder logits: {bad * 100:.3f}% out of tolerance, rel-L2 {rel:.3e}"


def test_inference_decoder_does_not_upsample_feature_maps(decoder, monkeypatch):
    from lavt_rs_b200 import _cabi as K
    _, dec = decoder
    calls = []
    for name in ("upsample_concat", "upsample_nhwc"):
        real = getattr(K, name)
        monkeypatch.setattr(K, name, lambda *a, _n=name, _r=real: (calls.append(_n), _r(*a))[1])
    c1, c2, c3, c4 = _feats(2, 32, seed=6)
    dec(c4.cuda(), c3.cuda(), c2.cuda(), c1.cuda())
    torch.cuda.synchronize()
    assert calls == [], f"inference decoder called {calls}"
