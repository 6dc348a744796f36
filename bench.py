#!/usr/bin/env python
"""Benchmark of the LAVT-RS hot path on B200:  python bench.py --gpus N --steps K --warmup W [--dump-outputs DIR]

Metric (BASELINE.json): LAVT-RS forward clips/s on 8x384x384 clips, Video Swin-B, 20-word expression.
One step = one ``LAVTVideo.forward(x, text ids, l_mask)`` (BERT-base text encoder + backbone + PWAM/gate + SimpleDecoding +
x4 upsample, every layer on the sm_100a kernels) over one batch of synthetic clips per GPU.

  value      whole-job clips/s, inputs resident in HBM, CUDA-graph replay of the forward, CUDA-event timed
  e2e        same metric through the public API call ``model(x, text, l_mask)`` with HOST (pinned) inputs:
             H2D of pixels / token ids / mask and D2H of the full-resolution logits inside the timed region
  roofline   the dominant kernel (tcgen05 GEMM / implicit-GEMM conv): algorithmic FLOPs / CUDA-event time vs the
             measured bf16 peak in MEASURED_PEAKS.json
  cpu_baseline / --impl reference   the oracle port of the reference forward (oracle/bert_oracle.py + oracle/lavt_oracle.py) timed on this
             box's host cores -- a reported baseline, not the target.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "LAVT-RS fwd clips/s (8x384^2)"
T_FRAMES, IMG, NL = 8, 384, 20


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=_positive, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write the logits of the last timed step to DIR/logits.npy as float32; an output "
                        "over 64 MB is cut to a seeded choice of whole frames, listed in the JSON line under dump_outputs.  With "
                        "WORLD_SIZE > 1 only rank 0's clips are written.  --impl reference times one clip of other inputs, so its "
                        "dump compares only with another --impl reference dump")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--clips-per-gpu", type=int, default=8)
    p.add_argument("--window12", action="store_true", help="(8,12,12) windows instead of the default (8,7,7)")
    p.add_argument("--sep-t-pwam", action="store_true",
                   help="the reference README's video configuration: SepTPWAM fusion (--sep_t_pwam --conv3d_kernel_size_t 3-3-3 "
                        "--conv3d_kernel_size_s 1-1-1 --w_t3x3_s1x1 --mm_t3x3_s1x1), 3118 GFLOP per clip")
    p.add_argument("--no-graph", action="store_true")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-extras", action="store_true",
                   help="skip the extra keys of the N=1 line: gpu_eager_baseline (the oracle port run as eager PyTorch on this GPU, fp32 and "
                        "bf16 autocast), latency_1clip (BASELINE configs[1] is literally one clip), window12 / sep_t_pwam throughput")
    return p.parse_args()


def _positive(s: str) -> int:
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1")
    return v


DUMP_BYTES = 64 * 10 ** 6


def dump_logits(out: torch.Tensor, d: str) -> dict:
    """Write ``out`` (n_frames, 2, H, W) as float32 to ``d``/logits.npy.  Over DUMP_BYTES, a seeded, sorted choice of whole frames is
    kept, so that two builds given the same arguments write the same frames."""
    import numpy as np
    n = out.shape[0]
    per_frame = out[0].numel() * 4
    keep = min(n, DUMP_BYTES // per_frame)
    frames = torch.arange(n) if keep == n else torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    arr = out[frames.to(out.device)].float().cpu().numpy()
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "logits.npy"), arr)
    return {"logits": {"shape": list(arr.shape), "of_shape": list(out.shape), "frames": frames.tolist()}}


SEP_T_PWAM = False      # set from --sep-t-pwam in main()
SEP_FLAGS = ["--sep_t_pwam", "--conv3d_kernel_size_t", "3-3-3", "--conv3d_kernel_size_s", "1-1-1", "--w_t3x3_s1x1", "--mm_t3x3_s1x1"]


def flops_per_clip(window12: bool) -> float:
    # BASELINE.md section 2 (measured with torch.utils.flop_counter on the reference), BERT-base (3.4 GFLOP) included;
    # SepTPWAM adds four Conv3d(3,3,3) per stage: +1043.6 GFLOP (3118.4 vs 2074.8 at window 8x7x7)
    return (2198.4e9 if window12 else 2074.8e9) + (1043.6e9 if SEP_T_PWAM else 0.0)


def model_args(window12: bool):
    from lavt_rs_b200.args import default_args
    return default_args(["--model", "lavt_video", "--swin_type", "base"] + (["--window12"] if window12 else [])
                        + (SEP_FLAGS if SEP_T_PWAM else []))


def build_model(window12: bool, device):
    from lavt_rs_b200.lib import segmentation
    torch.manual_seed(0)
    model = segmentation.lavt_video(pretrained="", args=model_args(window12))
    # the builder's init leaves LanguageGate live (init_weights overwrites the zero init, SURVEY.md TL;DR 3.5)
    return model.to(device).eval()


def synth_batch(B: int, seed: int):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, T_FRAMES, 3, IMG, IMG, generator=g)
    ids = torch.randint(1000, 5000, (B, NL), generator=g)      # token ids of a 20-word expression (SURVEY.md section 8d)
    m = torch.zeros(B, NL, dtype=torch.int64)
    m[:, :14] = 1
    return x, ids, m


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        self.t.join(timeout=2)
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [c.strip() for c in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def cpu_forward_time(window12: bool, sd_cpu, n_runs: int, threads: int):
    """Oracle port of the reference forward (BERT + backbone + decoder) on host cores: 1 clip per run."""
    from oracle import bert_oracle as BO
    from oracle import lavt_oracle as O
    torch.set_num_threads(threads)
    cfg = O.OracleConfig.swin("base", window12=window12, video=True)
    cfg.sep_t_pwam = SEP_T_PWAM
    x, l, m = synth_batch(1, 100)
    times, out = [], None
    with torch.no_grad():
        for _ in range(n_runs):
            t0 = time.perf_counter()
            l_feats = BO.bert_forward(sd_cpu, l, m).permute(0, 2, 1)        # lib/_utils.py:98-100
            out = O.model_forward(sd_cpu, cfg, x, l_feats, m)
            times.append(time.perf_counter() - t0)
    return times, out, (x, l, m)


def quick_throughput(model, B: int, dev, steps: int = 5, warmup: int = 3):
    """ms per forward of ``model`` over B device-resident clips (CUDA-graph replay, CUDA events, two rotating input batches)."""
    res = [tuple(t.to(dev) for t in synth_batch(B, 50 + s)) for s in range(2)]
    sx, sl, sm_ = (torch.empty_like(t) for t in res[0])
    with torch.no_grad():
        for t, r in zip((sx, sl, sm_), res[0]):
            t.copy_(r)
        model(sx, sl, sm_)
        torch.cuda.synchronize()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            model(sx, sl, sm_)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            model(sx, sl, sm_)

        def step(i):
            for t, r in zip((sx, sl, sm_), res[i % 2]):
                t.copy_(r)
            graph.replay()
        for i in range(warmup):
            step(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(i)
        e1.record()
        torch.cuda.synchronize()
    del graph
    return e0.elapsed_time(e1) / steps


def gpu_eager_baseline(window12: bool, sd_cpu, dev, B: int):
    """SURVEY.md section 8(d) / BASELINE.md section 4 call stock eager PyTorch on the same GPU "the real kernel to beat".  The Python
    reference cannot travel to the GPU box, so this leg runs its op-for-op restatement (the oracle port: same torch ops -- F.linear,
    softmax, F.conv2d / conv3d, F.layer_norm, ... -- dispatched to cuBLAS / cuDNN / ATen) on this GPU in fp32 and under bf16 autocast.
    Reported next to ``value``; it is a baseline leg like ``cpu_baseline`` and never part of the product path."""
    import contextlib
    from oracle import bert_oracle as BO
    from oracle import lavt_oracle as O
    cfg = O.OracleConfig.swin("base", window12=window12, video=True)
    cfg.sep_t_pwam = SEP_T_PWAM
    out = {"what": "oracle port of the reference forward as eager PyTorch (cuBLAS / cuDNN / ATen) on this GPU, BERT included",
           "tf32": bool(torch.backends.cuda.matmul.allow_tf32)}
    try:
        sd = {k: v.to(dev) for k, v in sd_cpu.items()}
    except Exception as e:                                  # noqa: BLE001
        out["error"] = repr(e)[:200]
        return out
    for name in ("fp32", "bf16_autocast"):
        for clips in dict.fromkeys((B, 1)):
            x, l, m = (t.to(dev) for t in synth_batch(clips, 100))
            ctx = torch.autocast("cuda", dtype=torch.bfloat16) if name == "bf16_autocast" else contextlib.nullcontext()
            try:
                with torch.no_grad(), ctx:
                    def fwd():
                        lf = BO.bert_forward(sd, l, m).permute(0, 2, 1)
                        return O.model_forward(sd, cfg, x, lf.float(), m)
                    fwd()
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    n = 3
                    for _ in range(n):
                        fwd()
                    e1.record()
                    torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / n
                out[f"{name}_{clips}clip"] = {"clips_per_s": clips / (ms * 1e-3), "ms_per_step": ms, "clips_per_step": clips}
            except Exception as e:                          # noqa: BLE001  (out of memory at 8 clips in fp32, unsupported op on CUDA, ...)
                out[f"{name}_{clips}clip"] = {"error": repr(e)[:200]}
                torch.cuda.empty_cache()
    return out


def train_step_extra(model, dev, world: int, rank: int, dist, clips: int = 4, steps: int = 5, warmup: int = 3):
    """BASELINE configs[3] next to the headline: one training step (BERT + backbone + decoder forward, weighted CE, hand-written backward,
    gradient all-reduce over NCCL launched per finished stage under the rest of the backward, SyncBN statistics) at ``clips`` clips per
    GPU.  Runs on EVERY rank (it contains collectives); returns the dict rank 0 reports under ``extras.train_step``."""
    from lavt_rs_b200 import engine as E
    from lavt_rs_b200 import train_engine as T
    from lavt_rs_b200 import training as TR
    # the steps below move the decoder's BatchNorm running statistics; they are put back afterwards so that the parity leg (which runs
    # later on the same model) still compares the model the headline number was measured on
    buffers = {k: v.detach().clone() for k, v in model.named_buffers()}
    drop_rates = [blk.drop_path_rate for layer in model.backbone.layers for blk in layer.blocks]
    model.train()
    for layer in model.backbone.layers:
        for blk in layer.blocks:
            blk.drop_path_rate = 0.0
    text = model.text_encoder
    text.eval()                                   # BERT dropout off: identical work, reproducible numbers
    params = [p for p in model.parameters() if p.requires_grad]
    seg_params = [p for p in list(model.backbone.parameters()) + list(model.classifier.parameters()) if p.requires_grad]
    batches = []
    for s_ in range(2):
        x, ids, m = synth_batch(clips, 201 + s_ + 10 * rank)
        g = torch.Generator().manual_seed(77 + s_ + 10 * rank)
        tgt = torch.randint(0, 2, (clips * T_FRAMES, IMG, IMG), generator=g)
        batches.append((x.to(dev), ids.to(dev), m.to(dev), tgt.to(dev)))
    state = {}

    # the text encoder (stock transformers module under autograd, ~600 tiny launches per direction) replays as two CUDA graphs on a side
    # stream under stage 0 of the hot path, like tools/bench_train.py; eager on the main stream if the capture is not possible
    text_fn = lambda ids_, m_: text(ids_, attention_mask=m_)[0].permute(0, 2, 1)       # noqa: E731  lib/_utils.py:98-100
    side = None
    try:
        text_fn = TR.GraphedTextEncoder(text, batches[0][1], batches[0][2])
        side = TR.SideStreamText(dev)
    except Exception as exc:       # noqa: BLE001
        print(f"train_step extra: text encoder not graph-captured ({type(exc).__name__}: {exc}); running it eagerly", file=sys.stderr)

    def step(i):
        x, ids, m, tgt = batches[i % 2]
        for p in params:
            p.grad = None
        grads = T.GradStore(seg_params)
        reducer = TR.GradReducer(overlap=True)
        if side is not None:
            l_feats, ready = side.forward(text_fn, ids, m)
            loss, dl = TR.segment_forward_backward(model, x, l_feats.detach(), m, tgt, grads, sync_bn=world > 1, on_ready=reducer.ready(grads),
                                                   lang_ready=ready, on_dl_ready=side.backward_hook())
            grads.finalize()
            side.join()
        else:
            l_feats = text_fn(ids, m)
            loss, dl = TR.segment_forward_backward(model, x, l_feats.detach(), m, tgt, grads, sync_bn=world > 1, on_ready=reducer.ready(grads))
            grads.finalize()
            l_feats.backward(dl)
        reducer.reduce([p for p in text.parameters() if p.requires_grad], grads)
        reducer.wait()
        state["loss"] = loss

    for i in range(warmup):
        step(i)
    E.LAUNCHES = 0
    step(0)
    launches = E.LAUNCHES
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if dist is not None:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    loss = float(state["loss"].item())
    for p in params:
        p.grad = None
    model.eval()
    with torch.no_grad():
        for k, v in model.named_buffers():
            v.copy_(buffers[k])
    for blk, r in zip([blk for layer in model.backbone.layers for blk in layer.blocks], drop_rates):
        blk.drop_path_rate = r
    return {"metric": "LAVT-RS train step clips/s (fwd+bwd, 8x384^2)", "clips_per_s": clips * world * steps / (ms * 1e-3), "ms_per_step": ms / steps,
            "n_gpus": world, "clips_per_gpu_per_step": clips, "steps": steps, "gpu_launches_per_step": launches, "loss": loss,
            "config": "BASELINE configs[3]: fwd + [0.9,1.1]-weighted CE + bwd in bf16, window 8x7x7, DropPath off, no optimizer update; "
                      + ("NCCL gradient all-reduce per finished stage under the rest of the backward (in place on the flat fp32 gradient "
                         "buffer, ReduceOp.AVG) + SyncBN statistics" if world > 1 else "single GPU: no collectives"),
            "peak_memory_bytes": torch.cuda.max_memory_allocated(dev)}


def run_reference(a):
    """--impl reference: the reference algorithm's CPU implementation (oracle port; the Python reference cannot travel)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    from lavt_rs_b200.lib import segmentation  # host modules only build parameters here (CPU); no kernels are run
    torch.manual_seed(0)
    model = segmentation.lavt_video(pretrained="", args=model_args(a.window12)).eval()
    sd = {k: v.detach().float() for k, v in model.state_dict().items()}
    warm = min(a.warmup, 1)
    cpu_forward_time(a.window12, sd, max(warm, 1), threads)
    steps = a.steps
    times, out, _ = cpu_forward_time(a.window12, sd, steps, threads)
    per = sum(times) / len(times)
    v = 1.0 / per
    sample = f"1 clip (8x384x384) per step, {steps} steps timed after {max(warm,1)} warm-up, fp32, torch CPU"
    dumped = dump_logits(out, a.dump_outputs) if a.dump_outputs else None
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "clips/s", "n_gpus": a.gpus, "steps": steps,
        "warmup": max(warm, 1), "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "LAVT-RS Video Swin-B forward (BERT-base text encoder + backbone + decoder), 8x384x384 clips, 20-token expression",
                   "window": "8x12x12" if a.window12 else "8x7x7", "clips_per_step": 1},
        "cpu_baseline": {"value": v, "unit": "clips/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        **({"dump_outputs": dumped} if dumped else {}),
    }))


def main():
    global SEP_T_PWAM
    a = parse()
    SEP_T_PWAM = bool(a.sep_t_pwam)
    if a.impl == "reference":
        return run_reference(a)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the B200 path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from lavt_rs_b200 import _cabi as K
    from lavt_rs_b200 import engine as E
    K.check(K.lib().lavt_check_device(), "lavt_check_device")

    B = a.clips_per_gpu
    model = build_model(a.window12, dev)
    # two rotating host batches (pinned) and their device-resident copies
    host = []
    for s in range(2):
        x, l, m = synth_batch(B, 1 + s + 10 * rank)
        host.append((x.pin_memory(), l.pin_memory(), m.pin_memory()))
    resident = [(x.to(dev), l.to(dev), m.to(dev)) for x, l, m in host]
    sx, sl, sm_ = (torch.empty_like(t) for t in resident[0])     # static graph inputs

    def fwd_static():
        return model(sx, sl, sm_)          # the reference's public call: LAVTVideo.forward(x, text ids, l_mask), BERT included

    with torch.no_grad():
        # eager warm-up (also builds bf16 weight copies, workspaces, func attributes)
        sx.copy_(resident[0][0]); sl.copy_(resident[0][1]); sm_.copy_(resident[0][2])
        E.LAUNCHES = 0
        out = fwd_static()
        launches_per_fwd = E.LAUNCHES
        torch.cuda.synchronize()
        graph = None
        if not a.no_graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                fwd_static()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = fwd_static()

        def step_resident(i):
            nonlocal out
            rx, rl, rm = resident[i % 2]
            sx.copy_(rx); sl.copy_(rl); sm_.copy_(rm)       # device-to-device refresh of the static inputs (part of the step)
            if graph is not None:
                graph.replay()                              # writes the captured ``out``
            else:
                out = fwd_static()

        host_out = torch.empty(out.shape, dtype=out.dtype).pin_memory()

        # e2e: three streams.  H2D of step i+1 and D2H of step i overlap the compute of the neighbouring steps; every
        # byte still crosses PCIe inside the timed region and the last D2H is waited for before the end event.
        h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
        stage = [tuple(torch.empty_like(t) for t in resident[0]) for _ in range(2)]
        out_stage = torch.empty_like(out)
        ev_h2d = [torch.cuda.Event() for _ in range(2)]
        ev_stage_free = [torch.cuda.Event() for _ in range(2)]
        ev_out_ready, ev_d2h_done = torch.cuda.Event(), torch.cuda.Event()
        e2e_state = {"primed": -1}

        def issue_h2d(i):
            b = i % 2
            with torch.cuda.stream(h2d_stream):
                h2d_stream.wait_event(ev_stage_free[b])
                for dst, src in zip(stage[b], host[b]):
                    dst.copy_(src, non_blocking=True)
                ev_h2d[b].record(h2d_stream)
            e2e_state["primed"] = i

        def step_e2e(i):
            cur = torch.cuda.current_stream()
            if e2e_state["primed"] != i:          # first step of a run: nothing was prefetched
                for b in range(2):
                    ev_stage_free[b].record(cur)
                ev_d2h_done.record(cur)
                issue_h2d(i)
            cur.wait_event(ev_h2d[i % 2])
            for dst, src in zip((sx, sl, sm_), stage[i % 2]):
                dst.copy_(src)                      # device-to-device into the graph's static inputs
            ev_stage_free[i % 2].record(cur)
            issue_h2d(i + 1)                        # next step's inputs travel while this step computes
            if graph is not None:
                graph.replay()
                o = out
            else:
                o = fwd_static()
            cur.wait_event(ev_d2h_done)             # previous step's result has left out_stage
            out_stage.copy_(o)
            ev_out_ready.record(cur)
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(ev_out_ready)
                host_out.copy_(out_stage, non_blocking=True)
                ev_d2h_done.record(d2h_stream)

        def finish_e2e():
            torch.cuda.current_stream().wait_event(ev_d2h_done)
            e2e_state["primed"] = -1

        def timed(step_fn, steps, warmup, finish=None):
            for i in range(warmup):
                step_fn(i)
            if finish is not None:
                finish()
            torch.cuda.synchronize()
            if dist is not None:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                step_fn(i)
            if finish is not None:
                finish()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            if dist is not None:
                t = torch.tensor([ms], device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dist.barrier()
                ms = t.item()
            return ms

        clocks = ClockSampler(local)
        if rank == 0:
            clocks.start()
        ms = timed(step_resident, a.steps, max(a.warmup, 3))
        clk = clocks.stop() if rank == 0 else None
        dumped = dump_logits(out, a.dump_outputs) if a.dump_outputs and rank == 0 else None
        ms_e2e = timed(step_e2e, a.steps, 1, finish_e2e)

        # --- roofline leg: per-launch CUDA events around the dominant kernel families (eager, same inputs) ---
        fam = None
        if rank == 0:
            K.TIMER.enabled = True
            K.TIMER.records.clear()
            fwd_static()
            _pk, _ = peaks()
            fam = K.TIMER.summary(_pk.get("bf16_tflops_sustained", 1400.0), _pk.get("hbm_gbs", 6550.0))
            K.TIMER.enabled = False

    train_extra = None
    if not a.no_extras and not a.window12 and not SEP_T_PWAM:
        try:
            train_extra = train_step_extra(model, dev, world, rank, dist)
        except Exception as e:                               # noqa: BLE001  (reported, never fatal for the headline line)
            train_extra = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    total_clips = B * world
    value = total_clips * a.steps / (ms * 1e-3)
    e2e_v = total_clips * a.steps / (ms_e2e * 1e-3)
    pk, pk_kind = peaks()
    g = fam.get("gemm_bf16_tc_kernel", {"launches": 0, "ms": 0.0, "flops": 0.0})
    at = fam.get("window_attn_kernel", {"launches": 0, "ms": 0.0, "flops": 0.0})
    achieved = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
    # DRAM bytes per launch of the dominant kernel: from the committed ncu capture of this same command (tools/ncu_r2.sh ->
    # profiles/r2_dram_traffic.json); used only when that capture saw the same number of launches per step as this run, else null
    traffic, traffic_src = None, None
    try:
        with open(os.path.join(ROOT, "profiles", "r2_dram_traffic.json")) as f:
            tj = json.load(f)["gemm_bf16_tc_kernel"]
        if not a.window12 and not SEP_T_PWAM and int(tj["launches_per_step"]) == int(g["launches"]):
            traffic = tj["dram_bytes_per_launch"]
            traffic_src = "profiles/r2_dram_traffic.json (ncu dram__bytes_read.sum + dram__bytes_write.sum over the %d launches of one step)" % g["launches"]
    except (OSError, KeyError, ValueError):
        pass
    roofline = {"kernel": "gemm_bf16_tc_kernel (tcgen05 GEMM + implicit-GEMM conv3x3)", "bound": "tensor",
                "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                "peak_kind": pk_kind + " sustained cuBLAS bf16", "traffic": traffic, "traffic_source": traffic_src,
                "alg_bytes_per_launch": (g.get("bytes") / g["launches"]) if g.get("bytes") and g["launches"] else None,
                "launches": g["launches"], "ms_per_step": g["ms"], "alg_flops_per_step": g["flops"],
                # per launch the binding roof is max(FLOPs / tensor peak, algorithmic bytes / HBM peak): short-K Swin
                # GEMMs (K = 128..256) are HBM-bound; this is sum(ideal) / sum(measured) over the step's launches
                "alg_bytes_per_step": g.get("bytes"), "frac_vs_binding_roof": (g["ideal_ms"] / g["ms"]) if g["ms"] > 0 else None,
                "attention_core": {"kernel": "window_attn_tc3_kernel (tcgen05/TMEM, 7x7 windows: row-parallel warpgroups, run-padded keys) / window_attn_tc2_kernel (tcgen05/TMEM key-chunked one-pass, other windows)",
                                   "impl": os.environ.get("LAVT_ATTN_IMPL", "auto"), "launches": at["launches"], "ms_per_step": at["ms"],
                                   "tflops": at["flops"] / (at["ms"] * 1e-3) / 1e12 if at["ms"] > 0 else 0.0},
                "whole_step_tflops": flops_per_clip(a.window12) * value / world / 1e12}

    h2d = sum(t.numel() * t.element_size() for t in host[0])
    d2h = host_out.numel() * host_out.element_size()
    res = {
        "metric": METRIC, "value": value, "unit": "clips/s", "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
        "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": {"workload": "LAVT-RS Video Swin-B forward (BERT-base text encoder + backbone + decoder), 8x384x384 clips, 20-token expression",
                   "window": "8x12x12" if a.window12 else "8x7x7", "fusion": "SepTPWAM (README video flags)" if SEP_T_PWAM else "PWAM",
                   "clips_per_gpu_per_step": B, "global_clips_per_step": total_clips,
                   "parallelism": f"clip-sharded x{world}, no collectives", "cuda_graph": graph is not None,
                   "l2": "two rotating input batches; per-step activations (>1 GB) exceed the 126 MB L2",
                   "flops_per_clip": flops_per_clip(a.window12)},
        "clocks": clk,
        "e2e": {"value": e2e_v, "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": launches_per_fwd * a.steps,
        "gpu_launches_per_step": launches_per_fwd,
        "roofline": roofline,
        "workspace_bytes": E.workspace(dev).bytes(),
    }
    if dumped:
        res["dump_outputs"] = dumped

    if world == 1 and not a.no_cpu_baseline:
        threads = os.cpu_count() or 1
        sd = {k: v.detach().float().cpu() for k, v in model.state_dict().items()}
        times, ref_out, (cx, cl, cm) = cpu_forward_time(a.window12, sd, 1, threads)
        with torch.no_grad():
            got = model(cx.to(dev), cl.to(dev), cm.to(dev)).float().cpu()
        rel = ((got - ref_out).norm() / ref_out.norm()).item()
        agree = (got.argmax(1) == ref_out.argmax(1)).float().mean().item()
        res["cpu_baseline"] = {"value": 1.0 / times[0], "unit": "clips/s", "cores": threads, "kind": "port",
                               "sample": "1 clip (8x384x384), 1 forward, fp32, oracle port of the reference on torch CPU"}
        err = (got - ref_out).abs().max().item()
        margin = (ref_out[:, 1] - ref_out[:, 0]).abs()
        clear = margin > 4 * err
        res["parity_vs_oracle"] = {"logits_rel_l2": rel, "argmax_agreement": agree, "max_abs_logit_err": err,
                                   "argmax_agreement_margin_filtered": (got.argmax(1) == ref_out.argmax(1))[clear].float().mean().item(),
                                   "margin_filter": "pixels whose fp32 |logit1 - logit0| exceeds 4x the max logit error",
                                   "pixels_kept": clear.float().mean().item()}
        if not a.no_extras:
            res["gpu_eager_baseline"] = gpu_eager_baseline(a.window12, sd, dev, B)
    if world == 1 and not a.no_extras:
        extras = {}
        with torch.no_grad():
            ms1 = quick_throughput(model, 1, dev, steps=10)
            extras["latency_1clip"] = {"ms": ms1, "clips_per_s": 1e3 / ms1, "config": "BASELINE configs[1]: one clip of 8x384x384, CUDA-graph replay"}
        del model
        torch.cuda.empty_cache()
        keep = SEP_T_PWAM
        for key, w12, sep in (("window12", True, False), ("sep_t_pwam", False, True)):
            if (w12, sep) == (a.window12, keep):
                continue
            try:
                SEP_T_PWAM = sep
                mdl = build_model(w12, dev)
                ms_x = quick_throughput(mdl, B, dev)
                extras[key] = {"clips_per_s": B / (ms_x * 1e-3), "ms_per_step": ms_x, "clips_per_step": B, "flops_per_clip": flops_per_clip(w12)}
                del mdl
                torch.cuda.empty_cache()
            except Exception as e:                          # noqa: BLE001
                extras[key] = {"error": repr(e)[:200]}
        SEP_T_PWAM = keep
        res["extras"] = extras
    if train_extra is not None:
        res.setdefault("extras", {})["train_step"] = train_extra
    print(json.dumps(res))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
