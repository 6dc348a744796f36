"""Attention-kernel micro-benchmark at the bench shapes (8 clips): python tools/bench_attn.py [impl ...]   (impl: auto tc2 tc3)"""
import math, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lavt_rs_b200 import _cabi as K
from lavt_rs_b200.geometry import window_geometry
def timeit(fn, iters=10, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters): fn()
    e.record(); torch.cuda.synchronize()
    return s.elapsed_time(e) / iters * 1e-3
impls = sys.argv[1:] or ["auto"]
for impl in impls:
    K.set_attention_impl(impl)
    for window in ((8, 7, 7), (8, 12, 12)):
        tot = 0.0
        for s, reps in ((0, 2), (1, 2), (2, 18), (3, 2)):
            for shifted in (False, True):
                C, nH, HW = 128 * 2 ** s, 4 * 2 ** s, 96 // 2 ** s
                geom = window_geometry(8, 8, HW, HW, window, shifted, True)
                rows = geom.rows()
                qkv = (torch.randn(rows, 3 * C, device="cuda") * 0.3).bfloat16()
                L = (2 * window[0] - 1) * (2 * window[1] - 1) * (2 * window[2] - 1)
                tt = (torch.randn(nH, L, device="cuda") * 0.5).contiguous()
                o = torch.empty(rows, C, device="cuda", dtype=torch.bfloat16)
                try:
                    t = timeit(lambda: K.window_attention(qkv, tt, geom, o))
                except Exception as ex:
                    print(f"[{impl}] window {window} stage {s}: {ex}")
                    continue
                print(f"[{impl}] window {window} stage {s} shifted {int(shifted)} N {geom.N}: {t*1e6:8.1f} us  {4.0*rows*geom.N*C/t/1e12:6.1f} TF   x{reps//2} = {t*reps/2*1e3:.3f} ms")
                tot += t * reps / 2
        print(f"[{impl}] window {window} total per step ms {tot * 1e3:.3f}")
