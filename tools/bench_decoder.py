"""Per-level A/B of the first conv of each SimpleDecoding level at the bench shapes (8 clips x 8 frames = 64 images, w7 model):
  old  upsample_concat + conv3x3(cat) + BN + ReLU                (the conv over the upsampled map)
  new  Z = W_tap . Y on the coarse map + conv3x3(skip) + upconv_blend  (engine._upconv_bn_relu)
Each repetition is timed alone with CUDA events after a 512 MB write that evicts L2 (126 MB), so the inputs come from HBM.
Prints the GPU name, power limit and SM clock read in the same run, and the max / rel-L2 difference of the two outputs.

    python tools/bench_decoder.py [--reps 20]
"""
import argparse
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from lavt_rs_b200 import _cabi as K            # noqa: E402
from lavt_rs_b200 import engine as E           # noqa: E402
from lavt_rs_b200.lib.mask_predictor import SimpleDecoding   # noqa: E402

N_IMG, HID = 64, 512
# (skip name, conv, bn, coarse side, coarse channels, fine side, skip channels)
LEVELS = [("c3", "conv1_4", "bn1_4", 12, 1024, 24, 512),
          ("c2", "conv1_3", "bn1_3", 24, HID, 48, 256),
          ("c1", "conv1_2", "bn1_2", 48, HID, 96, 128)]


def gpu_info() -> str:
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "nvidia-smi unavailable"


def timed(fn, reps: int, flush: torch.Tensor) -> float:
    """Median ms of ``reps`` single calls, each after an L2-evicting write."""
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    torch.manual_seed(0)
    dev = torch.device("cuda")
    dec = SimpleDecoding(1024, None)
    for m in dec.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.uniform_(0.5, 1.5)
            m.bias.data.uniform_(-0.2, 0.2)
            m.running_mean.uniform_(-0.2, 0.2)
            m.running_var.uniform_(0.5, 1.5)
    dec = dec.to(dev).eval()
    ws = E.Workspace()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    print(f"gpu: {gpu_info()}")
    tot_old = tot_new = 0.0
    for skip_name, conv, bn, h, cy, H, cs in LEVELS:
        y = torch.randn(N_IMG, h, h, cy, device=dev).to(torch.bfloat16)
        skip = torch.randn(N_IMG, H, H, cs, device=dev).to(torch.bfloat16)
        cat = torch.empty(N_IMG, H, H, cy + cs, device=dev, dtype=torch.bfloat16)
        t_old = torch.empty(N_IMG, H, H, HID, device=dev, dtype=torch.bfloat16)
        t_new = torch.empty_like(t_old)

        def old():
            K.upsample_concat(y, skip, cat)
            E._cbr(cat, dec, conv, bn, t_old)

        def new():
            E._upconv_bn_relu(y, skip, dec, conv, bn, ws, t_new)

        ms_old, ms_new = timed(old, args.reps, flush), timed(new, args.reps, flush)
        old()
        new()
        torch.cuda.synchronize()
        d = (t_new.float() - t_old.float())
        rel = (d.norm() / t_old.float().norm()).item()
        fl_old = 2.0 * N_IMG * H * H * HID * 9 * (cy + cs)
        fl_new = 2.0 * N_IMG * (h * h * 9 * HID * cy + H * H * HID * 9 * cs)
        print(f"{H}x{H} ({conv}, {cy}+{cs} -> {HID}): old {ms_old:.3f} ms ({fl_old / 1e12:.2f} TF)  new {ms_new:.3f} ms "
              f"({fl_new / 1e12:.2f} TF)  new/old {ms_new / ms_old:.3f}   max|diff| {d.abs().max().item():.3e}  rel-L2 {rel:.3e}")
        # the three pieces of the new path on the buffers and prepared weights it just used
        z, p = ws.get("dec_z", (N_IMG, h, h, 9 * HID), torch.bfloat16, dev), ws.get("dec_p", (N_IMG, H, H, HID), torch.float32, dev)
        wy, (s, b) = dec.prepared._cache[conv + "_up"][1], dec.prepared._cache[bn][1]
        w_s = dec.prepared._cache[conv + "_skip"][1]
        ms_z = timed(lambda: K.gemm_bf16(y.view(-1, cy), wy, out_bf16=z.view(-1, 9 * HID)), args.reps, flush)
        ms_s = timed(lambda: K.conv3x3_bf16(skip, w_s, cscale=s, bias=b, out_f32=p.view(-1, HID)), args.reps, flush)
        ms_b = timed(lambda: K.upconv_blend(z, p, s, b, t_new), args.reps, flush)
        gb = (z.numel() * 2 + p.numel() * 4 + t_new.numel() * 2) / 1e9
        print(f"   new pieces: Z gemm {ms_z:.3f} ms  skip conv {ms_s:.3f} ms  blend {ms_b:.3f} ms ({gb:.2f} GB, {gb / ms_b:.2f} TB/s)")
        tot_old += ms_old
        tot_new += ms_new
    print(f"sum of levels: old {tot_old:.3f} ms  new {tot_new:.3f} ms  saved {tot_old - tot_new:.3f} ms")
    print(f"gpu after: {gpu_info()}")


if __name__ == "__main__":
    main()
