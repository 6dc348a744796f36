#!/usr/bin/env python
"""Training-step benchmark (BASELINE config 4): LAVT-RS Video Swin-B, fwd + weighted CE + bwd in bf16 on the sm_100a kernels,
4 clips (8x384x384) per GPU, gradient all-reduce over NCCL at N > 1.

    python tools/bench_train.py --steps 5 --warmup 2
    python tools/bench_train.py --window12 --graph           # the (8,12,12)-window model (attention backward on attn_bwd_tc2.cu)
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/bench_train.py --gpus 2

One step = what the reference's ``train_one_epoch_ytvos`` does per iteration up to the optimizer (train.py:430-470):
``optimizer.zero_grad(); output = model(image, text, l_mask); loss = criterion(output, target); loss.backward()`` plus DDP's
gradient all-reduce.  The text encoder runs as the stock ``transformers`` module under autograd (its input gradient comes from the
kernels); DropPath is disabled (SURVEY.md section 8d, config 4).  Prints one JSON line (same keys as bench.py where they apply).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench as B0  # noqa: E402  (shared helpers: synthetic batch, clocks, peaks)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--clips-per-gpu", type=int, default=4)
    p.add_argument("--frozen-text", action="store_true", help="do not backpropagate into the text encoder")
    p.add_argument("--optimizer", action="store_true", help="include the AdamW update (FusedAdamW over the reference's parameter groups, "
                                                            "poly LR) in the timed step")
    p.add_argument("--window12", action="store_true", help="(8,12,12) windows instead of the default (8,7,7)")
    p.add_argument("--sep-t-pwam", action="store_true", help="the reference README's video configuration (SepTPWAM fusion flags)")
    p.add_argument("--no-overlap-allreduce", dest="overlap_allreduce", action="store_false",
                   help="all-reduce after the backward instead of launching each stage's all-reduce under the rest of the backward (default)")
    p.add_argument("--bf16-allreduce", action="store_true", help="cast the gradient buckets to bf16 for the all-reduce")
    p.add_argument("--graph", action="store_true", help="capture forward + loss + backward of the hot path (everything after the text encoder) "
                                                        "in one CUDA graph (1 GPU only: SyncBN / gradient collectives stay eager)")
    p.add_argument("--serial-text", action="store_true", help="text encoder forward / backward on the main stream, before / after the hot path, "
                   "instead of on a side stream under stage 0 (default)")
    p.add_argument("--eager-text", action="store_true", help="run the text encoder eagerly instead of as CUDA graphs")
    p.add_argument("--phases", action="store_true", help="print CUDA-event times of the phases of one step to stderr")
    p.add_argument("--by-tag", action="store_true", help="print the CUDA-event time of every GEMM / attention shape of one step to stderr")
    p.add_argument("--cpu-baseline", action="store_true", help="also time the oracle's fwd+bwd of one clip on the host cores (~1 min, 14 GB)")
    a = p.parse_args()

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    from lavt_rs_b200 import _cabi as K
    from lavt_rs_b200 import engine as E
    from lavt_rs_b200 import train_engine as T
    from lavt_rs_b200 import training as TR
    K.check(K.lib().lavt_check_device(), "lavt_check_device")

    B0.SEP_T_PWAM = bool(a.sep_t_pwam)
    model = B0.build_model(a.window12, dev).train()
    for layer in model.backbone.layers:
        for blk in layer.blocks:
            blk.drop_path_rate = 0.0
    text = model.text_encoder
    text.eval()          # BERT dropout off: the timed work is identical, the numbers reproducible
    for prm in text.parameters():
        prm.requires_grad_(not a.frozen_text)
    params = [prm for prm in model.parameters() if prm.requires_grad]

    opt = sched = None
    if a.optimizer:
        from lavt_rs_b200.optim import FusedAdamW, poly_lr_lambda, reference_param_groups
        opt = FusedAdamW(reference_param_groups(model, "encoder-10"), lr=5e-5, weight_decay=1e-2, amsgrad=True)    # args.py defaults
        sched = torch.optim.lr_scheduler.LambdaLR(opt, poly_lr_lambda(100000))

    Bc = a.clips_per_gpu
    batches = []
    for s in range(2):
        x, ids, m = B0.synth_batch(Bc, 1 + s + 10 * rank)
        g = torch.Generator().manual_seed(77 + s + 10 * rank)
        tgt = torch.randint(0, 2, (Bc * B0.T_FRAMES, B0.IMG, B0.IMG), generator=g)
        batches.append((x.to(dev), ids.to(dev), m.to(dev), tgt.to(dev)))

    state = {}
    text_fn = lambda ids, m: text(ids, attention_mask=m)[0].permute(0, 2, 1)             # noqa: E731  lib/_utils.py:98-100
    if not a.eager_text and not a.frozen_text:
        text_fn = TR.GraphedTextEncoder(text, batches[0][1], batches[0][2])

    graph_state = {}

    def build_graph():
        """Static-input CUDA graph of segment_forward_backward: ~1000 short launches replayed without Python / launch gaps."""
        x0, ids0, m0, tgt0 = batches[0]
        gs = graph_state
        gs["x"], gs["m"], gs["tgt"] = x0.clone(), m0.clone(), tgt0.clone()
        gs["l"] = torch.zeros(x0.shape[0], 768, ids0.shape[1], device=dev)
        seg_params = [prm for prm in list(model.backbone.parameters()) + list(model.classifier.parameters()) if prm.requires_grad]
        for prm in seg_params:
            prm.grad = None
        for mod in model.modules():           # bf16 weight copies must be (re)built INSIDE the capture so that every replay refreshes them
            if hasattr(mod, "prepared"):
                mod.prepared.clear()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):         # one eager pass on the capture stream: workspaces, function attributes
            TR.segment_forward_backward(model, gs["x"], gs["l"], gs["m"], gs["tgt"], T.GradStore(seg_params))
        torch.cuda.current_stream().wait_stream(side)
        for mod in model.modules():
            if hasattr(mod, "prepared"):
                mod.prepared.clear()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            grads = T.GradStore(seg_params)
            gs["loss"], gs["dl"] = TR.segment_forward_backward(model, gs["x"], gs["l"], gs["m"], gs["tgt"], grads)
            grads.finalize()                  # param.grad = views of the graph-owned flat buffer (zeroed by the captured memset)
        gs["graph"] = g

    def step_graph(i):
        x, ids, m, tgt = batches[i % 2]
        gs = graph_state
        for prm in text.parameters():
            prm.grad = None
        l_feats = text_fn(ids, m)
        gs["x"].copy_(x); gs["m"].copy_(m); gs["tgt"].copy_(tgt); gs["l"].copy_(l_feats.detach())
        gs["graph"].replay()
        if not a.frozen_text:
            l_feats.backward(gs["dl"])
        if opt is not None:
            opt.step()
            sched.step()
        state["loss"] = gs["loss"]

    def step(i):
        if graph_state.get("graph") is not None and not K.TIMER.enabled:
            return step_graph(i)
        x, ids, m, tgt = batches[i % 2]
        for prm in params:
            prm.grad = None                                                    # optimizer.zero_grad(set_to_none=True)
        grads = T.GradStore(params)
        reducer = TR.GradReducer(overlap=a.overlap_allreduce, compress="bf16" if a.bf16_allreduce else None)
        if a.serial_text or a.frozen_text or K.TIMER.enabled:
            l_feats = text_fn(ids, m)
            loss, dl = TR.segment_forward_backward(model, x, l_feats.detach(), m, tgt, grads, sync_bn=world > 1, on_ready=reducer.ready(grads))
            grads.finalize()
            if not a.frozen_text:
                l_feats.backward(dl)
        else:
            # text encoder forward / backward on a side stream, under stage 0 of the hot path (TR.SideStreamText)
            side = state.setdefault("side", TR.SideStreamText(dev))
            l_feats, ready = side.forward(text_fn, ids, m)
            loss, dl = TR.segment_forward_backward(model, x, l_feats.detach(), m, tgt, grads, sync_bn=world > 1, on_ready=reducer.ready(grads),
                                                   lang_ready=ready, on_dl_ready=side.backward_hook())
            grads.finalize()
            side.join()
        if not a.frozen_text:
            reducer.reduce([prm for prm in text.parameters() if prm.requires_grad], grads)
        reducer.wait()
        if opt is not None:
            opt.step()
            sched.step()
        state["loss"] = loss

    def timed(steps, warmup):
        for i in range(warmup):
            step(i)
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
        return ms

    if a.phases and rank == 0:
        def ev():
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            return e
        for _ in range(3):
            step(0)
        x, ids, m, tgt = batches[0]
        for prm in params:
            prm.grad = None
        marks = [("start", ev())]
        l_feats = text_fn(ids, m)
        marks.append(("text encoder forward (torch)", ev()))
        logits, tape = TR.segment_forward(model, x, l_feats.detach(), m, sync_bn=False)
        marks.append(("segment forward (saved activations)", ev()))
        acc = torch.zeros(2, device=dev)
        K.cross_entropy(logits, tgt, acc, phase=0)
        dlog = torch.empty_like(logits)
        K.cross_entropy(logits, tgt, acc, dlog, phase=1)
        marks.append(("weighted cross-entropy fwd + bwd", ev()))
        grads = T.GradStore()
        stage_marks = []
        dl = TR.segment_backward(model, tape, dlog, grads, on_ready=lambda ps: stage_marks.append(ev()))
        marks.append(("segment backward", ev()))
        grads.finalize()
        marks.append(("hand gradients to param.grad", ev()))
        if not a.frozen_text:
            l_feats.backward(dl)
        marks.append(("text encoder backward (torch autograd)", ev()))
        if opt is not None:
            opt.step()
        marks.append(("FusedAdamW", ev()))
        torch.cuda.synchronize()
        for (n0, e0), (n1, e1) in zip(marks, marks[1:]):
            print(f"{e0.elapsed_time(e1):8.2f} ms  {n1}", file=sys.stderr)
        names = ["decoder backward", "stage 3 backward", "stage 2 backward", "stage 1 backward", "stage 0 backward", "patch embed backward"]
        prev = marks[3][1]
        for nm, e in zip(names, stage_marks):
            print(f"    {prev.elapsed_time(e):8.2f} ms  {nm}", file=sys.stderr)
            prev = e
    E.LAUNCHES = 0
    step(0)
    torch.cuda.synchronize()
    launches = E.LAUNCHES
    if a.graph:
        if world > 1:
            raise SystemExit("--graph is a 1-GPU option")
        build_graph()
    peak_mem = torch.cuda.max_memory_allocated(dev)
    clocks = B0.ClockSampler(local)
    if rank == 0:
        clocks.start()
    ms = timed(a.steps, max(a.warmup, 3))
    clk = clocks.stop() if rank == 0 else None

    # roofline leg: per-launch CUDA events on rank 0; EVERY rank runs the step (it contains collectives)
    fam = None
    K.TIMER.enabled = rank == 0
    K.TIMER.records.clear()
    step(0)
    torch.cuda.synchronize()
    if rank == 0:
        pk, pk_kind = B0.peaks()
        fam = K.TIMER.summary(pk.get("bf16_tflops_sustained", 1400.0), pk.get("hbm_gbs", 6550.0))
        if a.by_tag:
            for (f_, tag), d in sorted(K.TIMER.by_tag().items(), key=lambda kv: -kv[1]["ms"]):
                print(f"{d['ms']:8.3f} ms  x{d['launches']:3d}  {d['flops'] / max(d['ms'], 1e-9) / 1e9:7.0f} TFLOP/s  {f_}  {tag}", file=sys.stderr)
    K.TIMER.enabled = False
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    total = Bc * world
    value = total * a.steps / (ms * 1e-3)
    flops_clip = 3.0 * (B0.flops_per_clip(a.window12) - 3.4e9)          # forward + input gradients + weight gradients of every contraction
    g = fam.get("gemm_bf16_tc_kernel", {"launches": 0, "ms": 0.0, "flops": 0.0})
    ab = fam.get("window_attn_bwd_kernel", {"launches": 0, "ms": 0.0, "flops": 0.0})
    af = fam.get("window_attn_kernel", {"launches": 0, "ms": 0.0, "flops": 0.0})
    peak = pk.get("bf16_tflops_sustained", pk.get("bf16_tflops"))
    achieved = g["flops"] / (g["ms"] * 1e-3) / 1e12 if g["ms"] > 0 else 0.0
    res = {
        "metric": "LAVT-RS train step clips/s (fwd+bwd, 8x384^2)", "value": value, "unit": "clips/s", "n_gpus": world, "steps": a.steps,
        "warmup": max(a.warmup, 3), "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "LAVT-RS Video Swin-B training step: BERT-base + backbone + decoder forward, [0.9,1.1]-weighted CE, backward, "
                               "gradient all-reduce; 8x384x384 clips, 20-token expression, window " + ("8x12x12" if a.window12 else "8x7x7") + ", DropPath off, no optimizer update",
                   "clips_per_gpu_per_step": Bc, "global_clips_per_step": total,
                   "parallelism": f"data-parallel x{world}" + ((", NCCL gradient all-reduce (" + ("per stage, under the backward" if a.overlap_allreduce else "after the backward") + ") + SyncBN statistics") if world > 1 else ""),
                   "text_encoder": "frozen" if a.frozen_text else ("transformers BertModel under autograd (fp32)" + ("" if a.eager_text else ", forward and backward replayed as CUDA graphs")),
                   "cuda_graph": bool(a.graph), "l2": "two rotating batches; saved activations (> 10 GB) exceed the 126 MB L2", "flops_per_clip": flops_clip},
        "clocks": clk, "loss": float(state["loss"].item()), "gpu_launches": launches * a.steps, "gpu_launches_per_step": launches,
        "peak_memory_bytes": peak_mem,
        "roofline": {"kernel": "gemm_bf16_tc_kernel (forward GEMMs / convs, input-gradient GEMMs / convs, split-K weight-gradient GEMMs)",
                     "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if peak else None,
                     "peak_kind": pk_kind + " sustained cuBLAS bf16", "traffic": None, "launches": g["launches"], "ms_per_step": g["ms"],
                     "alg_flops_per_step": g["flops"],
                     "attention_bwd": {"kernel": "window_attn_bwd_tc_kernel (tcgen05 / TMEM; 7 x 7 windows with saved row statistics) / window_attn_bwd_kernel (mma.sync, windows that fit its shared memory) / window_attn_bwd_tc2_kernel (tcgen05 / TMEM; larger windows, e.g. 8 x 12 x 12)", "launches": ab["launches"], "ms_per_step": ab["ms"],
                                       "tflops": ab["flops"] / (ab["ms"] * 1e-3) / 1e12 if ab["ms"] > 0 else 0.0},
                     "attention_fwd": {"launches": af["launches"], "ms_per_step": af["ms"]},
                     "whole_step_tflops": flops_clip * value / world / 1e12},
    }
    if a.cpu_baseline and world == 1:
        from oracle import lavt_oracle as O
        torch.set_num_threads(os.cpu_count() or 1)
        cfg = O.OracleConfig.swin("base", window12=a.window12, video=True)
        sd = {k: v.detach().float().cpu().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in model.state_dict().items()}
        x, ids, m = B0.synth_batch(1, 100)
        tgt = torch.randint(0, 2, (B0.T_FRAMES, B0.IMG, B0.IMG))
        l = torch.randn(1, 768, B0.NL)
        t0 = time.perf_counter()
        out = O.model_forward(sd, cfg, x, l, m, train_bn=True)
        O.weighted_cross_entropy(out, tgt).backward()
        dt = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": 1.0 / dt, "unit": "clips/s", "cores": os.cpu_count(), "kind": "port",
                               "sample": "1 clip (8x384x384), 1 fwd+bwd after BERT, fp32, autograd through the oracle port on torch CPU"}
    print(json.dumps(res))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
