"""Window-attention core (C-ABI lavt_window_attention) in isolation vs a plain fp32 PyTorch evaluation of the same op on
the same bf16 q/k/v (SURVEY.md Appendix B shapes: every distinct N the kernel must support).  bias index and shift mask of
the torch side come from the host geometry (tests/test_geometry.py pins that bit-exactly to the reference).
Tolerance: |a-b| <= 2e-2*|b| + 2e-2*rms(b), rel-L2 <= 1e-2 (P is rounded to bf16 before P.V; fp32 accumulation)."""
import math

import pytest
import torch

pytestmark = pytest.mark.gpu


def torch_window_attention(qkv, table, geom):
    """qkv bf16 [rows, 3C] (q pre-scaled by hd^-0.5*log2e); table fp32 [L, nH] -> fp32 [rows, C]"""
    from lavt_rs_b200.geometry import rel_const, window_row_map
    rows, C3 = qkv.shape
    C = C3 // 3
    nH = table.shape[1]
    N = geom.N
    nwin = rows // N
    _, code, rid = window_row_map(geom)
    code, rid = code.cuda().view(nwin, N), rid.cuda().view(nwin, N)
    x = (qkv if qkv.dtype == torch.float64 else qkv.float()).view(nwin, N, 3, nH, 32).permute(2, 0, 3, 1, 4)
    q, k, v = x[0] / math.log2(math.e), x[1], x[2]
    s = q @ k.transpose(-1, -2)
    idx = code[0][:, None] - code[0][None, :] + rel_const(geom)
    s = s + table[idx.reshape(-1)].view(N, N, nH).permute(2, 0, 1).unsqueeze(0)
    if geom.sd or geom.sh or geom.sw:
        s = s + ((rid[:, :, None] != rid[:, None, :]).to(s.dtype) * -100.0).unsqueeze(1)
    return (s.softmax(-1) @ v).transpose(1, 2).reshape(rows, C)


CASES = [  # (B, D, H, W), window, shifted, heads
    ((1, 8, 14, 14), (8, 7, 7), True, 4), ((1, 8, 96, 96), (8, 7, 7), True, 4), ((1, 4, 24, 24), (8, 7, 7), True, 16),
    ((1, 16, 14, 14), (8, 7, 7), True, 8), ((1, 8, 24, 24), (8, 12, 12), True, 16), ((1, 4, 48, 48), (8, 12, 12), True, 8),
    ((1, 8, 12, 12), (8, 12, 12), True, 32), ((1, 16, 24, 24), (8, 12, 12), True, 16), ((2, 1, 30, 30), (1, 12, 12), True, 8),
    ((2, 1, 15, 15), (1, 7, 7), True, 32), ((1, 8, 10, 10), (8, 12, 12), True, 4), ((3, 8, 14, 21), (8, 7, 7), False, 4),
    # attn_tc3.cu corner cases: a two-frame window (N = 98, one partial tile), a single (window, head) unit, and enough units per CTA that the
    # K / V stages, the Q ring and the bias table (several heads per CTA) all wrap around
    ((1, 2, 14, 14), (8, 7, 7), True, 4), ((1, 8, 7, 7), (8, 7, 7), False, 1), ((4, 8, 24, 24), (8, 7, 7), True, 16),
    # clamped windows of fewer than 16 tokens (mma.sync fallback): N = 4, 8, 6, a single token, the 12 x 12 table, N = 14 shifted along h
    ((1, 4, 1, 1), (8, 7, 7), True, 4), ((1, 8, 1, 1), (8, 7, 7), True, 8), ((2, 3, 1, 2), (8, 7, 7), True, 32),
    ((1, 1, 1, 1), (8, 7, 7), False, 4), ((2, 2, 2, 3), (8, 12, 12), True, 16), ((1, 1, 14, 2), (8, 7, 7), True, 4),
    # the smallest attn_tc2.cu windows (N = 16 shifted along d, 30)
    ((1, 16, 2, 1), (8, 7, 7), True, 4), ((2, 2, 3, 5), (8, 7, 7), True, 8),
    # clamped windows of 48 ... 400 tokens: stage 3 of the video models at 8 x 192^2 (w7, N = 288), 8 x 160^2 (w7 and w12, N = 200) and
    # 4 x 320^2 (w12, N = 400), shorter clips, and a window clamped along w only (shift and mask along h)
    ((1, 8, 6, 6), (8, 7, 7), True, 32), ((2, 8, 5, 5), (8, 7, 7), True, 32), ((1, 4, 6, 6), (8, 7, 7), True, 16),
    ((1, 8, 3, 3), (8, 7, 7), True, 8), ((1, 8, 14, 5), (8, 7, 7), True, 4), ((1, 8, 5, 5), (8, 12, 12), True, 32),
    ((1, 4, 10, 10), (8, 12, 12), True, 32),
]


# auto = attn_tc3.cu for full 7 x 7 / 12 x 12 windows (row-parallel warpgroups, run-padded keys), attn_tc2.cu for the other windows of 16+
# tokens, the mma.sync kernel below that; tc2 = the one-pass chunked tcgen05 kernel wherever it applies (N >= 16)
@pytest.mark.parametrize("impl", ["auto", "tc2"])
@pytest.mark.parametrize("dims,window,shifted,nH", CASES)
def test_window_attention_matches_torch(dims, window, shifted, nH, impl):
    from lavt_rs_b200 import _cabi as K
    from lavt_rs_b200.geometry import window_geometry
    B, D, H, W = dims
    clamp = window[0] != 1
    geom = window_geometry(B, D, H, W, window, shifted, clamp)
    C = nH * 32
    rows = geom.rows()
    g = torch.Generator(device="cuda").manual_seed(rows + nH)
    qkv = torch.randn(rows, 3 * C, device="cuda", generator=g)
    qkv[:, :C] *= 32 ** -0.5 * math.log2(math.e) * 2.0        # scores with a few units of spread
    qkv = qkv.bfloat16()
    L = (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)
    table = torch.randn(L, nH, device="cuda", generator=g)
    out = torch.empty(rows, C, device="cuda", dtype=torch.bfloat16)
    prev = K.set_attention_impl(impl)
    try:
        K.window_attention(qkv, table.t().contiguous(), geom, out)
        torch.cuda.synchronize()
    finally:
        K.set_attention_impl(prev)
    ref = torch_window_attention(qkv, table, geom)
    err = (out.float() - ref).abs()
    rms = ref.pow(2).mean().sqrt()
    bad = (err > 2e-2 * ref.abs() + 2e-2 * rms).float().mean().item()
    rel = (err.norm() / ref.norm()).item()
    assert bad < 1e-4 and rel < 1e-2, f"N={geom.N}: {bad*100:.4f}% out of tolerance, rel-L2 {rel:.3e}"


@pytest.mark.parametrize("dims,window,nH", [((1, 8, 14, 14), (8, 7, 7), 4), ((1, 8, 24, 24), (8, 12, 12), 4), ((1, 4, 24, 24), (8, 7, 7), 4),
                                            ((1, 8, 10, 10), (8, 12, 12), 4)])
@pytest.mark.parametrize("pattern", ["ramp", "spike", "late_rows"])
@pytest.mark.parametrize("impl", ["tc2", "tc3"])
def test_one_pass_softmax_slow_path(dims, window, nH, pattern, impl):
    """The one-pass kernel keeps the running maximum of the FIRST piece of a row and only re-bases when a later piece overflows
    sum 2^(s - m) <= 2^20.  These inputs force that slow path: scores that grow by hundreds of units along the key axis ('ramp'),
    a single huge key in the last chunk ('spike': rescale of the P columns already written AND of the O accumulator in TMEM), and
    rows whose maximum moves only for part of a warp ('late_rows')."""
    from lavt_rs_b200 import _cabi as K
    from lavt_rs_b200.geometry import window_geometry
    B, D, H, W = dims
    geom = window_geometry(B, D, H, W, window, True, True)
    C = nH * 32
    rows, N = geom.rows(), geom.N
    g = torch.Generator(device="cuda").manual_seed(7)
    qkv = torch.randn(rows, 3 * C, device="cuda", generator=g)
    qkv[:, :C] *= 32 ** -0.5 * math.log2(math.e)
    t = torch.arange(rows, device="cuda") % N
    # feature 0 of q / k carries the forced score: s_ij += q_i0 * k_j0
    if pattern == "ramp":
        qkv[:, 0] = 4.0
        qkv[:, C] = (t.float() / N) * 150.0                 # + up to 600 log2-units from the first to the last key
    elif pattern == "spike":
        qkv[:, 0] = 4.0
        qkv[:, C] = torch.where(t == N - 3, 120.0, 0.0)
    else:
        qkv[:, 0] = torch.where(t % 5 == 0, 4.0, 0.0)       # only every fifth query row sees the ramp
        qkv[:, C] = (t.float() / N) * 100.0
    qkv = qkv.bfloat16()
    L = (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)
    table = torch.randn(L, nH, device="cuda", generator=g)
    out = torch.empty(rows, C, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(rows, nH, device="cuda", dtype=torch.float32)
    prev = K.set_attention_impl(impl)       # tc3 = auto: attn_tc2.cu for the windows that are not full 7 x 7 / 12 x 12
    try:
        K.window_attention(qkv, table.t().contiguous(), geom, out, lse=lse)
        torch.cuda.synchronize()
    finally:
        K.set_attention_impl(prev)
    ref = torch_window_attention(qkv, table, geom)
    err = (out.float() - ref).abs()
    rms = ref.pow(2).mean().sqrt()
    bad = (err > 2e-2 * ref.abs() + 2e-2 * rms).float().mean().item()
    rel = (err.norm() / ref.norm()).item()
    assert torch.isfinite(out.float()).all() and torch.isfinite(lse).all()
    assert bad < 1e-4 and rel < 1e-2, f"{pattern} N={N}: {bad*100:.4f}% out of tolerance, rel-L2 {rel:.3e}"
