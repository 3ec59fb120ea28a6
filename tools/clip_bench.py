"""Throughput of the GPU clip pipeline (SURVEY.md 8 f-2) at the pretraining batch size, next to the Pillow oracle on the
host cores (one process, as one DataLoader worker would run it).
    python tools/clip_bench.py [B] [--size S] [--frames T] [--views pretrain|finetune] [--ab-lib PATH]

--size / --frames set the clip geometry (default 16 x 112 x 112); --views finetune times one-view finetune training
clips (FinetuneClipSampler.plan_train) instead of the two pretraining views.  "layout" in the output is the launch
layout of the batch: CTAs per (frame, view) and shared memory per CTA.  --ab-lib PATH times this tree's
`cstp_clip_assemble` against the one exported by another build of the library (same descriptor layout) on the same
uploaded descriptors, alternating the two over 10 rounds of 20 launches each."""
import argparse
import ctypes as C
import json
import os
import random
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cstp_b200 import lib as L  # noqa: E402
from cstp_b200.data_process.clip_plan import FinetuneClipSampler, PretrainClipSampler  # noqa: E402
from cstp_b200.data_process.gpu_clips import GpuClipPipeline, clip_layout, collate_labels  # noqa: E402
from cstp_b200.synthetic import synthetic_video  # noqa: E402
from oracle.clip_oracle import render_plan, render_view  # noqa: E402  (only for the Pillow CPU timing leg below)

ap = argparse.ArgumentParser()
ap.add_argument("B", nargs="?", type=int, default=60)
ap.add_argument("--size", type=int, default=112)
ap.add_argument("--frames", type=int, default=16)
ap.add_argument("--views", choices=("pretrain", "finetune"), default="pretrain")
ap.add_argument("--ab-lib", default=None)
args = ap.parse_args()
B, S, T = args.B, args.size, args.frames
W, H, F = 320, 240, 150
random.seed(0)
np.random.seed(0)
torch.manual_seed(0)
host_vids = [synthetic_video(F + 1, W, H, b % 4) for b in range(4)]
vids = [torch.from_numpy(host_vids[b % 4]).cuda() for b in range(B)]
pipe = GpuClipPipeline(T, S)
if args.views == "pretrain":
    sampler = PretrainClipSampler(T, S)
    draw, run, n_views = (lambda: sampler.plan(F, W, H)), pipe.assemble, 2
else:
    sampler = FinetuneClipSampler(T, S)
    draw, run, n_views = (lambda: sampler.plan_train(F, W, H)), pipe.assemble_clips, 1
views_of = (lambda p: p.views) if n_views == 2 else (lambda p: (p.view,))
out = None
t_plan, t_gpu = [], []
a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
for it in range(8):
    t0 = time.perf_counter()
    plans = [draw() for _ in range(B)]
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    a.record()
    out = run(plans, vids, out)
    if n_views == 2:
        labels = collate_labels(plans, device="cuda")
    b_.record()
    torch.cuda.synchronize()
    t2 = time.perf_counter()
    if it >= 3:
        t_plan.append(t1 - t0)
        t_gpu.append((a.elapsed_time(b_), t2 - t1))
from torch.profiler import ProfilerActivity, profile  # noqa: E402
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    out = run(plans, vids, out)
    torch.cuda.synchronize()
kern_us = sum(e.device_time for e in prof.events() if "clip_assemble" in e.name)
max_h = max(H if v.resize is not None else v.box[3] - v.box[1] for p in plans for v in views_of(p))
# Pillow oracle on the host: 4 samples
t0 = time.perf_counter()
for i in range(4):
    if n_views == 2:
        render_plan(plans[i], host_vids[i % 4], S)
    else:
        render_view(plans[i].view, host_vids[i % 4], plans[i].frame_base, S)
cpu_per_sample = (time.perf_counter() - t0) / 4
res = {"B": B, "frame": [W, H], "views": args.views, "sample_duration": T, "sample_size": S,
       "layout": dict(zip(("ctas_per_frame_view", "smem_bytes_per_cta"), clip_layout(S, max_h))), "max_crop_h": max_h,
       "plan_ms_per_batch": 1e3 * float(np.mean(t_plan)),
       "kernel_ms_per_batch": kern_us / 1e3, "in_bytes_touched_per_batch": int(sum(
           (v.box[2] - v.box[0]) * (v.box[3] - v.box[1]) * 3 * T for p in plans for v in views_of(p))),
       "gpu_ms_per_batch_events": float(np.mean([g[0] for g in t_gpu])),
       "host_wall_ms_per_batch": 1e3 * float(np.mean([g[1] for g in t_gpu])),
       "samples_per_s_gpu": B / (float(np.mean([g[1] for g in t_gpu])) + float(np.mean(t_plan))),
       "pillow_cpu_ms_per_sample_1core": 1e3 * cpu_per_sample, "samples_per_s_pillow_1core": 1.0 / cpu_per_sample,
       "out_bytes_per_batch": n_views * B * 3 * T * S * S * 4}
if args.ab_lib:
    other = C.CDLL(os.path.abspath(args.ab_lib))
    libs = {"this": L.load(), "other": other}
    for lib in libs.values():
        lib.cstp_clip_assemble.restype, lib.cstp_clip_assemble.argtypes = L.SIGNATURES["cstp_clip_assemble"]
    buf = pipe._stage[n_views * B]                 # the descriptors and tables of the last batch, still on the device
    stream = torch.cuda.current_stream().cuda_stream
    ms = {k: [] for k in libs}
    for rnd in range(10):
        for k in (("this", "other") if rnd % 2 == 0 else ("other", "this")):
            L.check(libs[k].cstp_clip_assemble(buf["ddesc"].data_ptr(), n_views * B, T, S, max_h, stream))
            torch.cuda.synchronize()
            a.record()
            for _ in range(20):
                L.check(libs[k].cstp_clip_assemble(buf["ddesc"].data_ptr(), n_views * B, T, S, max_h, stream))
            b_.record()
            torch.cuda.synchronize()
            ms[k].append(a.elapsed_time(b_) / 20)
    res["ab_kernel_ms_per_batch"] = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "max": float(np.max(v)),
                                         "rounds": v} for k, v in ms.items()}
print(json.dumps(res))
