"""Window-attention backward: the tcgen05 kernels (attn_bwd_tc.cu, attn_bwd_tc2.cu) and the mma.sync kernel (attn_bwd.cu) vs float64
autograd, and their timing.
    python tools/run_attn_bwd.py [--bench [--w12]] [--case i]
--bench times the 7 x 7 stage shapes (mma / tc / forced tc2), --bench --w12 the four 8 x 12 x 12 stage shapes of 4 clips at 384^2 (tc2: the
only kernel for N = 1152) and clamped w12 windows both tc2 and the mma.sync kernel can run."""
import math
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lavt_rs_b200 import _cabi as K  # noqa: E402
from lavt_rs_b200.geometry import window_geometry  # noqa: E402


def torch_window_attention(qkv, table, geom):
    """same evaluation as tests/test_attention_gpu.py: qkv [rows, 3C] (q pre-scaled by hd^-0.5 * log2 e), table [L, nH] -> [rows, C]"""
    from lavt_rs_b200.geometry import rel_const, window_row_map
    rows, C3 = qkv.shape
    C = C3 // 3
    nH = table.shape[1]
    N = geom.N
    nwin = rows // N
    _, code, rid = window_row_map(geom)
    code, rid = code.cuda().view(nwin, N), rid.cuda().view(nwin, N)
    x = qkv.view(nwin, N, 3, nH, 32).permute(2, 0, 3, 1, 4)
    q, k, v = x[0] / math.log2(math.e), x[1], x[2]
    s = q @ k.transpose(-1, -2)
    idx = code[0][:, None] - code[0][None, :] + rel_const(geom)
    s = s + table[idx.reshape(-1)].view(N, N, nH).permute(2, 0, 1).unsqueeze(0)
    if geom.sd or geom.sh or geom.sw:
        s = s + ((rid[:, :, None] != rid[:, None, :]).to(s.dtype) * -100.0).unsqueeze(1)
    return (s.softmax(-1) @ v).transpose(1, 2).reshape(rows, C)


CASES = [((1, 8, 14, 14), True, 4), ((1, 4, 14, 14), True, 4), ((1, 2, 14, 14), True, 4), ((1, 8, 7, 7), False, 1), ((3, 8, 14, 21), False, 4),
         ((4, 8, 24, 24), True, 16), ((1, 6, 21, 14), True, 8)]
BENCH = [((4, 8, 96, 96), True, 4), ((4, 8, 48, 48), True, 8), ((4, 8, 24, 24), True, 16), ((4, 8, 24, 24), False, 16), ((4, 8, 12, 12), True, 32)]
W12 = (8, 12, 12)
# (dims, shifted, heads, window, kernels to time): the four stage shapes of the --window12 model (4 clips, 8 x 384^2: N = 1152 everywhere),
# then clamped w12 windows of 400 (4 x 10 x 10) and 288 (2 x 12 x 12) tokens that the mma.sync kernel can run too
BENCH_W12 = [((4, 8, 96, 96), True, 4, W12, ("tc2",)), ((4, 8, 48, 48), True, 8, W12, ("tc2",)), ((4, 8, 24, 24), True, 16, W12, ("tc2",)),
             ((4, 8, 12, 12), True, 32, W12, ("tc2",)), ((64, 4, 10, 10), True, 8, W12, ("mma", "tc2")),
             ((32, 2, 24, 24), True, 8, W12, ("mma", "tc2"))]


def rel(a, b):
    return ((a.float() - b.float()).norm() / (b.float().norm() + 1e-20)).item()


def setup(dims, shifted, nH, seed=0, window=(8, 7, 7)):
    B, D, H, W = dims
    geom = window_geometry(B, D, H, W, tuple(window), shifted, True)
    L = (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)
    C = nH * 32
    rows = geom.rows()
    g = torch.Generator(device="cuda").manual_seed(rows + nH + seed)
    qkv = torch.randn(rows, 3 * C, device="cuda", generator=g)
    qkv[:, :C] *= 32 ** -0.5 * math.log2(math.e) * 2.0
    qkv = qkv.bfloat16()
    table = torch.randn(L, nH, device="cuda", generator=g)
    dout = torch.randn(rows, C, device="cuda", generator=g).bfloat16()
    out = torch.empty(rows, C, device="cuda", dtype=torch.bfloat16)
    lse = torch.empty(rows, nH, device="cuda", dtype=torch.float32)
    K.window_attention(qkv, table.t().contiguous(), geom, out, lse=lse)
    return geom, qkv, table, dout, out, lse


def run(impl, geom, qkv, table, dout, out, lse):
    prev = K.set_attention_bwd_impl(impl)
    try:
        dqkv = torch.zeros_like(qkv)
        dtab = torch.zeros(table.shape[1], table.shape[0], device="cuda")
        K.window_attention_bwd(qkv, out, dout, table.t().contiguous(), geom, dqkv, dtab, lse=lse)
        torch.cuda.synchronize()
    finally:
        K.set_attention_bwd_impl(prev)
    return dqkv, dtab


def reference(geom, qkv, table, dout):
    C = qkv.shape[1] // 3
    x = qkv.double().requires_grad_(True)
    t = table.double().requires_grad_(True)
    o = torch_window_attention(x, t, geom)
    o.backward(dout.double())
    dq = x.grad.clone()
    # the kernels return the gradient of the UNSCALED projection output: y_q = q' / (hd^-0.5 log2 e)
    dq[:, :C] *= 32 ** -0.5 * math.log2(math.e)
    return dq, t.grad.t().contiguous()


def main():
    if "--bench" in sys.argv:
        shapes = BENCH_W12 if "--w12" in sys.argv else [(d, s, h, (8, 7, 7), ("mma", "tc", "tc2")) for d, s, h in BENCH]
        for dims, shifted, nH, window, impls in shapes:
            geom, qkv, table, dout, out, lse = setup(dims, shifted, nH, window=window)
            tt = table.t().contiguous()
            dqkv = torch.zeros_like(qkv)
            dtab = None if "--notab" in sys.argv else torch.zeros(nH, table.shape[0], device="cuda")
            res = {}
            for impl in impls:
                prev = K.set_attention_bwd_impl(impl)
                nws = K.window_attention_bwd_workspace_floats(tt, geom)       # under the selection just made
                ws = torch.empty(nws, device="cuda") if nws > 0 else None
                for _ in range(2):
                    K.window_attention_bwd(qkv, out, dout, tt, geom, dqkv, dtab, lse=lse, workspace=ws)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(20):
                    K.window_attention_bwd(qkv, out, dout, tt, geom, dqkv, dtab, lse=lse, workspace=ws)
                e1.record()
                torch.cuda.synchronize()
                K.set_attention_bwd_impl(prev)
                res[impl] = e0.elapsed_time(e1) / 20 * 1e3
            rows = geom.rows()
            fl = 10.0 * rows * geom.N * nH * 32
            times = "  ".join(f"{k} {v:.1f} us ({fl / v / 1e6:.0f} TFLOP/s)" for k, v in res.items())
            print(f"{dims} window={window} N={geom.N} shifted={shifted} nH={nH}: {times}", flush=True)
        return
    cases = CASES
    if "--case" in sys.argv:
        cases = [CASES[int(sys.argv[sys.argv.index("--case") + 1])]]
    ok = True
    for dims, shifted, nH in cases:
        geom, qkv, table, dout, out, lse = setup(dims, shifted, nH)
        C = nH * 32
        ref_q, ref_t = reference(geom, qkv, table, dout)
        for impl in ("mma", "tc"):
            dqkv, dtab = run(impl, geom, qkv, table, dout, out, lse)
            e = [rel(dqkv[:, i * C:(i + 1) * C], ref_q[:, i * C:(i + 1) * C]) for i in range(3)] + [rel(dtab, ref_t)]
            good = all(x < 2e-2 for x in e)
            ok = ok and good
            print(f"{dims} shifted={shifted} nH={nH} N={geom.N} {impl}: dq {e[0]:.2e} dk {e[1]:.2e} dv {e[2]:.2e} dtable {e[3]:.2e} {'ok' if good else 'FAIL'}", flush=True)
    print("ALL OK" if ok else "FAILED")


if __name__ == "__main__":
    main()
