"""BASELINE config 4: r21d finetune step (batch 60, 101-way head) and batch-1 test-mode inference latency on one B200.
    python tools/finetune_bench.py [--sample-size S] [--sample-duration T] [--batch B] [--test-videos N]
        > finetune_bench.json

--sample-size / --sample-duration set the clip geometry (default 16 x 112 x 112).  When batch B does not fit in device
memory at that geometry, the step is timed at the largest smaller multiple of 4 that does ("batch" in the output says
which).  --test-videos N also times cstp_b200.evaluate.test_videos at that geometry over N seeded 171x128 videos."""
import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cstp_b200.models.pace.r21d_byol import R21DBYOL  # noqa: E402
from cstp_b200 import ops  # noqa: E402


def timed(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = ops.launch_count()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (ops.launch_count() - n0) / iters


ap = argparse.ArgumentParser()
ap.add_argument("--sample-size", type=int, default=112)
ap.add_argument("--sample-duration", type=int, default=16)
ap.add_argument("--batch", type=int, default=60)
ap.add_argument("--test-videos", type=int, default=0)
args = ap.parse_args()
T, S = args.sample_duration, args.sample_size
out = {"sample_duration": T, "sample_size": S}
g = torch.Generator().manual_seed(0)
m = None
for B in range(args.batch, 0, -4):
    try:
        torch.manual_seed(1)
        m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda().train()
        x = (torch.rand(B, 3, T, S, S, generator=g) * 2 - 1).cuda()
        y = torch.randint(0, 101, (B,), generator=g).cuda()
        torch.cuda.reset_peak_memory_stats()
        ms, launches = timed(lambda: m.finetune_step(x, y, lr=0.025, momentum=0.9, weight_decay=1e-3), 10)
        break
    except torch.OutOfMemoryError:
        m = x = y = None
        torch.cuda.empty_cache()
flops = B * (3 * 42.733e9 - 1.224e9) * (T * S * S) / (16 * 112 * 112)   # SURVEY.md 8(d): 3F - 1.224 GFLOP per 16x112 clip
out["finetune_step_b60"] = {"batch": B, "ms_per_step": ms, "clips_per_s": B / ms * 1e3, "launches_per_step": launches,
                            "step_tflops": flops / ms / 1e9, "peak_allocated_bytes": torch.cuda.max_memory_allocated()}
m.eval()
for b in (1, 10):
    xb = x[:b].contiguous()
    with torch.no_grad():
        ms, launches = timed(lambda: m(xb, None, o_type="test"), 30, warm=5)
    out[f"test_latency_b{b}"] = {"ms": ms, "clips_per_s": b / ms * 1e3, "launches": launches}
if args.test_videos:
    from cstp_b200.data_process.datasets import GpuVideoStore  # noqa: E402
    from cstp_b200.evaluate import test_videos  # noqa: E402
    del x
    gl = torch.Generator().manual_seed(1)
    frames = torch.randint(60, 400, (args.test_videos,), generator=gl).tolist()
    labels = torch.randint(0, 101, (args.test_videos,), generator=gl).tolist()
    store = GpuVideoStore()
    gd = torch.Generator(device="cuda").manual_seed(0)
    for v, f in enumerate(frames):
        store.put(v, torch.randint(0, 256, (f, 128, 171, 3), dtype=torch.uint8, device="cuda", generator=gd))
    passes = []
    for _ in range(4):                            # the first pass builds the inference engines and is not counted
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = test_videos(m, store, frames, labels, sample_duration=T, sample_size=S)
        torch.cuda.synchronize()
        passes.append(time.perf_counter() - t0)
    t = sorted(passes[1:])[1]
    out["test_videos"] = {"videos": r["videos"], "clips": r["clips"], "pass_s": passes[1:], "videos_per_s": r["videos"] / t,
                          "clips_per_s": r["clips"] / t}
print(json.dumps(out))
