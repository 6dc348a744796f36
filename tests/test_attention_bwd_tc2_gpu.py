"""Window-attention backward on attn_bwd_tc2.cu (tcgen05 / TMEM, key tiles outer, dQ partials through an fp32 workspace): every window
of 16 ... 1152 tokens, against float64 autograd through a plain PyTorch evaluation of the same op on the same bf16 q / k / v / dO (the
helpers of tools/run_attn_bwd.py), and against the other two kernels where they apply.  Tolerance: rel-L2 <= 1e-2 per gradient, as for
the other backward kernels (bf16 operands and outputs, fp32 accumulation)."""
import importlib.util
import os

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W7, W12 = (8, 7, 7), (8, 12, 12)


def _tool():
    spec = importlib.util.spec_from_file_location("run_attn_bwd", os.path.join(ROOT, "tools", "run_attn_bwd.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _check(t, geom, qkv, table, dout, dqkv, dtab, what, tol=1e-2):
    C = qkv.shape[1] // 3
    ref_q, ref_t = t.reference(geom, qkv, table, dout)
    errs = {"dq": t.rel(dqkv[:, :C], ref_q[:, :C]), "dk": t.rel(dqkv[:, C:2 * C], ref_q[:, C:2 * C]),
            "dv": t.rel(dqkv[:, 2 * C:], ref_q[:, 2 * C:]), "dtable": t.rel(dtab, ref_t)}
    assert all(e < tol for e in errs.values()), f"{what} N={geom.N}: {errs}"
    return errs


# (B, D, H, W), shifted, heads, window.  w12: N = 1152 (unshifted, H/W-shifted, and D/H/W-shifted with a 16-frame clip), 576, clamped
# 800 (8 x 10 x 10) and 648 (8 x 9 x 9), several windows / heads / units per CTA.  Forced tc2 on w7: N = 392 / 196, a clamped 4 x 6 x 5 = 120
# (one key tile, no workspace) and small / clamped windows of 16 ... 400 tokens (2 x 2 x 4, 1 x 5 x 6, 8 x 7 x 5, 8 x 5 x 10, 4 x 10 x 10).
CASES = [
    ((1, 8, 24, 24), False, 4, W12), ((1, 8, 24, 24), True, 4, W12), ((1, 16, 24, 24), True, 8, W12), ((2, 4, 24, 24), True, 4, W12),
    ((1, 8, 10, 10), False, 8, W12), ((1, 8, 9, 9), True, 4, W12), ((3, 8, 36, 36), True, 16, W12), ((1, 8, 12, 12), True, 32, W12),
    ((1, 8, 14, 14), True, 4, W7), ((1, 4, 14, 14), True, 4, W7), ((4, 8, 24, 24), True, 16, W7), ((2, 4, 6, 5), False, 4, W7),
    ((1, 2, 2, 4), False, 4, W7), ((3, 1, 5, 6), True, 4, W7), ((2, 8, 14, 5), True, 4, W7), ((1, 8, 5, 10), False, 4, W12),
    ((2, 4, 10, 10), True, 8, W12),
]


@pytest.mark.parametrize("dims,shifted,nH,window", CASES)
def test_tc2_matches_autograd(dims, shifted, nH, window):
    from lavt_rs_b200 import _cabi as K
    t = _tool()
    geom, qkv, table, dout, out, lse = t.setup(dims, shifted, nH, window=window)
    prev = K.set_attention_bwd_impl("tc2")
    try:
        assert K.window_attention_bwd_kernel(table.t(), geom) == "tc2"
    finally:
        K.set_attention_bwd_impl(prev)
    dqkv, dtab = t.run("tc2", geom, qkv, table, dout, out, lse)
    _check(t, geom, qkv, table, dout, dqkv, dtab, f"{dims} shifted={shifted} nH={nH} window={window}")


# kernel against kernel on shapes both run: tc on full 7 x 7 windows, mma on windows that fit its shared memory.  Each kernel is held to
# float64 autograd above; their mutual distance is bounded by twice their own bf16 error.
PAIRS = [((1, 8, 14, 14), True, 4, W7, "tc"), ((3, 8, 14, 21), False, 4, W7, "tc"), ((2, 2, 14, 14), True, 8, W7, "tc"),
         ((2, 4, 10, 10), True, 8, W12, "mma"), ((4, 2, 24, 24), True, 4, W12, "mma"), ((2, 8, 14, 5), True, 4, W7, "mma")]


@pytest.mark.parametrize("dims,shifted,nH,window,other", PAIRS)
def test_tc2_agrees_with_the_other_kernels(dims, shifted, nH, window, other):
    t = _tool()
    geom, qkv, table, dout, out, lse = t.setup(dims, shifted, nH, window=window)
    C = nH * 32
    ref_q, ref_t = t.reference(geom, qkv, table, dout)
    d2, t2 = t.run("tc2", geom, qkv, table, dout, out, lse)
    d1, t1 = t.run(other, geom, qkv, table, dout, out, lse)
    for name, sl in (("dq", slice(0, C)), ("dk", slice(C, 2 * C)), ("dv", slice(2 * C, 3 * C))):
        own = t.rel(d1[:, sl], ref_q[:, sl])
        assert t.rel(d2[:, sl], d1[:, sl]) <= 2 * own + 1e-4, (name, t.rel(d2[:, sl], d1[:, sl]), own)
    own = t.rel(t1, ref_t)
    assert t.rel(t2, t1) <= 2 * own + 1e-4, ("dtable", t.rel(t2, t1), own)


def test_tc2_table_gradient_accumulates_and_may_be_null():
    """dtable_t accumulates (+=) across calls; NULL skips it and leaves dqkv unchanged; a caller-owned workspace and the one the binding
    allocates give the same result; a workspace that is too small is refused."""
    from lavt_rs_b200 import _cabi as K
    t = _tool()
    geom, qkv, table, dout, out, lse = t.setup((2, 8, 24, 24), True, 4, window=W12)
    tt = table.t().contiguous()
    d1, tab1 = t.run("tc2", geom, qkv, table, dout, out, lse)
    need = K.window_attention_bwd_workspace_floats(tt, geom)
    assert need >= 1152 * 32
    ws = torch.full((need,), float("nan"), device="cuda")      # not read across calls: stale contents do not matter
    acc = tab1.clone()
    dq2 = torch.zeros_like(qkv)
    K.window_attention_bwd(qkv, out, dout, tt, geom, dq2, acc, lse=lse, workspace=ws)
    torch.cuda.synchronize()
    assert t.rel(acc, 2 * tab1) < 1e-3
    assert torch.equal(dq2, d1)
    dq3 = torch.zeros_like(qkv)
    K.window_attention_bwd(qkv, out, dout, tt, geom, dq3, None, lse=lse, workspace=ws)
    torch.cuda.synchronize()
    assert torch.equal(dq3, d1)
    with pytest.raises(K.LavtError):
        K.window_attention_bwd(qkv, out, dout, tt, geom, dq3, None, lse=lse, workspace=ws[:1000])
