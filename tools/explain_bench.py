"""Grad-CAM throughput of cstp_b200.explain at batch 64 on 16 x 112 x 112 clips, against the same Grad-CAM through torch
autograd on oracle/cstp_oracle.finetune_forward(training=False) on the same GPU (fp32 with TF32 off, and under bf16
autocast, as tests/torch_gpu_bar.py runs stock PyTorch).

    python tools/explain_bench.py [--out profiles/r11_explain_bench.json] [--iters 5] [--rounds 3]

Reported: clips/s of class_activation_maps for every stage and with input_grad (graph-replayed, host clock around
synchronised calls, median of --rounds rounds of --iters calls), the same for torch, peak max_memory_allocated of each
(reset before it), and the CAM kernels' own time (cam_seed, gradcam, cam_upsample) from CUDA events around standalone
launches on the engine's buffers.  The card's name, power limit and maximum SM clock are read in the same run."""
from __future__ import annotations

import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, T, S = 64, 16, 112
STAGES = ("conv2", "conv3", "conv4", "conv5")
TORCH_CHUNK = 16         # clips per torch autograd call: a batch of 64 does not fit the card's 180 GB in fp32


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(fn, iters, rounds):
    out = []
    for _ in range(rounds):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(iters):
            fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) / iters * 1e3)
    med = statistics.median(out)
    return {"median_ms": med, "spread_ms": max(out) - min(out), "clips_per_s": B / med * 1e3}


def peak(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() / 2 ** 30


def release(m):
    """Frees the model's cached engines (their closures hold reference cycles, so the collector has to run)."""
    m.free_inference_engines()
    gc.collect()
    torch.cuda.empty_cache()


def torch_cam(state, x, stage, amp):
    """Grad-CAM through autograd on the oracle's eval forward: the stage output is caught at its ReLU."""
    from oracle import cstp_oracle as O
    idx = {"conv2": 5, "conv3": 10, "conv4": 15, "conv5": 20}[stage]
    seen = []

    class _Relu:
        def __getattr__(self, k):
            return getattr(F, k)

        @staticmethod
        def relu(t):
            seen.append(F.relu(t))
            return seen[-1]
    saved, O.F = O.F, _Relu()
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
            logits, _ = O.finetune_forward(state, x, training=False)
    finally:
        O.F = saved
    A = seen[idx]
    score = logits.float().gather(1, logits.float().argmax(1, keepdim=True)).sum()
    (dA,) = torch.autograd.grad(score, [A])
    alpha = dA.float().mean(dim=(2, 3, 4))
    cam = F.relu((alpha[:, :, None, None, None] * A.float()).sum(1))
    cam = F.interpolate(cam[:, None], size=(T, S, S), mode="trilinear", align_corners=False)[:, 0]
    lo, hi = cam.flatten(1).min(1).values, cam.flatten(1).max(1).values
    return (cam - lo[:, None, None, None]) / (hi - lo).clamp_min(1e-30)[:, None, None, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_explain_bench.json"))
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("explain_bench measures the B200 path: it needs a CUDA device")
    from cstp_b200 import ops
    from cstp_b200.explain import class_activation_maps
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(0)
    m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda().eval()
    x = torch.randn(B, 3, T, S, S, device="cuda")
    res = {"batch": B, "clip": [T, S, S], **card(), "measured": True}
    ours = {}
    for stage in STAGES:
        for ig in (False, True) if stage == "conv5" else (False,):
            name = stage + ("+input_grad" if ig else "")
            fn = lambda: class_activation_maps(m, x, stage=stage, input_grad=ig)      # noqa: E731
            fn()
            ours[name] = timed(fn, a.iters, a.rounds)
            ours[name]["peak_gib"] = peak(fn)
            release(m)                                 # one engine resident at a time, as a user with one setting has
    res["cstp_b200"] = ours
    # CAM kernels alone, on the conv2 (largest) and conv5 engine buffers
    kern = {}
    for stage in ("conv2", "conv5"):
        class_activation_maps(m, x, stage=stage)
        eng = next(e for k, e in m._infer.items() if k[0] == "explain" and k[5] == stage)
        launches = {
            "cam_seed": lambda: ops.cam_seed(eng.logits, B, 101, None, eng.classes, eng.dlogits),
            "gradcam": lambda: ops.gradcam(eng.stage_act, eng.stage_grad, B, eng.stage_channels, eng.alpha, eng.cam_small),
            "cam_upsample": lambda: ops.cam_upsample(eng.cam_small, B, eng.cam),
        }
        for kname, fn in launches.items():
            for _ in range(3):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(50):
                fn()
            e1.record()
            torch.cuda.synchronize()
            kern[f"{stage}.{kname}_us"] = e0.elapsed_time(e1) / 50 * 1e3
        del eng, launches, fn
        release(m)
    res["cam_kernels"] = kern
    # stock PyTorch autograd on the oracle's eval forward, same weights
    state = {k: v for k, v in m.state_dict().items()}
    xt = x.clone().requires_grad_(True)
    ref = {}
    for amp in (False, True):
        for stage in ("conv2", "conv5"):
            fn = lambda: [torch_cam(state, xt[i:i + TORCH_CHUNK], stage, amp) for i in range(0, B, TORCH_CHUNK)]  # noqa: E731
            r = timed(fn, a.iters, a.rounds)
            r["peak_gib"] = peak(fn)
            ref[("bf16_autocast." if amp else "fp32.") + stage] = r
    res["torch_autograd"] = ref
    res["torch_autograd_chunk"] = TORCH_CHUNK
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
