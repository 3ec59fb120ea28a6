"""Optimiser launches and the fused pretraining step with SGD, Adam and AdamW on one B200.

    python tools/optim_bench.py [--out profiles/r08_optim_bench.json] [--steps 10] [--warmup 3]

1. The optimiser launch (clip-norm pass + update kernel: cstp_sgd_clip_step / cstp_adam_clip_step, clipping on) on the
   flat buffers of the pretraining model (25.43 M parameters) and of the UCF101 finetune model: mean ms per launch over at
   least 1 s of back-to-back launches (CUDA events) after a warm-up; the pretraining buffers (102 MB each, 814 MB per Adam launch)
   exceed the 126 MB L2 together; the finetune model's are 58 MB each, so its launches are partly served from L2.  A separate torch.profiler pass gives each kernel's own time.
   Bytes per parameter: the norm pass reads g (4 B); the SGD update reads p, g, momentum and writes p, momentum (20 B);
   the Adam update reads p, g, exp_avg, exp_avg_sq and writes p, exp_avg, exp_avg_sq (28 B).  Achieved GB/s are those
   bytes over the measured time; the share is against the 6.55 TB/s of HBM bandwidth measured on a B200 (DESIGN.md).
2. The fused batch-60 pretraining step (R21DBYOL.train_step, 16x112x112 clips resident in HBM, the captured CUDA graph)
   with each optimiser: mean step time and samples/s over --steps timed steps after --warmup, and the peak of allocated
   device memory.
The card's name and power limit are read in the same run.  Prints one JSON line and writes it to --out."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.test_eval_bench import card  # noqa: E402

HBM_TBS = 6.55
MIN_TIMED_S = 1.0
LOSS_WEIGHT = (0.1, 1.0, 1.0, 1.0, 1.0)
UPDATE_BYTES = {"sgd": 20, "adam": 28, "adamw": 28}
NORM_BYTES = 4


def timed(fn, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, total = 0, 0.0
    while total < MIN_TIMED_S * 1e3:
        n = max(1, calls)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        calls += n
    return total / calls, calls


def launcher(kind, n):
    from cstp_b200 import ops
    from cstp_b200.engine import adam_scalars
    g = torch.Generator(device="cuda").manual_seed(1)
    p = torch.randn(n, device="cuda", generator=g) * 0.05
    gr = torch.randn(n, device="cuda", generator=g) * 1e-3
    s1, s2 = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    norm_out, ws = torch.zeros(2, device="cuda"), torch.zeros(2048, device="cuda")
    if kind == "sgd":
        return lambda: ops.sgd_clip_step(p, gr, s1, 1e-3, 0.9, 5e-4, 18.0, True, False, norm_out, ws)
    h = adam_scalars(10, 1e-3, (0.9, 0.999), 1e-8, 5e-4, kind == "adamw", 18.0, True)
    return lambda: ops.adam_clip_step(p, gr, s1, s2, h, norm_out, ws)


def kernel_times(fn, reps=20):
    """Per-kernel mean device time (ms) of fn's launches, from a torch.profiler pass of its own."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and "kernel" in e.key:
            name = e.key.split("(")[0].split("::")[-1]
            out[name] = getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) / 1e3 / reps
    return out


def optimiser_launches():
    from cstp_b200.engine import FlatStore, trainable_param_specs
    from cstp_b200.engine_ft import finetune_param_specs
    sizes = {"pretrain": FlatStore(trainable_param_specs(), "meta").numel,
             "finetune_ucf101": FlatStore(finetune_param_specs(101, True), "meta").numel}
    res = {}
    for where, n in sizes.items():
        for kind in ("sgd", "adam", "adamw"):
            fn = launcher(kind, n)
            ms, calls = timed(fn)
            kt = kernel_times(fn)
            upd = kt.get("sgd_step_kernel" if kind == "sgd" else "adam_step_kernel")
            norm = kt.get("sumsq_partial_kernel")
            b_launch = (NORM_BYTES + UPDATE_BYTES[kind]) * n
            b_upd = UPDATE_BYTES[kind] * n
            res[f"{where}/{kind}"] = {
                "params": n, "launch_ms": ms, "launches_timed": calls, "bytes_per_launch": b_launch,
                "launch_gbs": b_launch / ms / 1e6, "launch_share_of_6p55": b_launch / ms / 1e9 / HBM_TBS,
                "update_kernel_ms": upd, "norm_kernel_ms": norm, "update_kernel_bytes": b_upd,
                "update_kernel_gbs": b_upd / upd / 1e6 if upd else None,
                "update_kernel_share_of_6p55": b_upd / upd / 1e9 / HBM_TBS if upd else None,
                "update_kernel_floor_ms": b_upd / (HBM_TBS * 1e9)}
            del fn
            torch.cuda.empty_cache()
    return res


def step_rates(steps, warmup, B=60):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    res = {}
    for kind in ("sgd", "adam", "adamw"):
        torch.manual_seed(1)
        m = R21DBYOL(pretrain=True).cuda()
        g = torch.Generator(device="cuda").manual_seed(2)
        x1 = torch.rand(B, 3, 16, 112, 112, device="cuda", generator=g)
        x2 = torch.rand(B, 3, 16, 112, 112, device="cuda", generator=g)
        labels = tuple(torch.randint(0, 5, (B,), device="cuda", generator=g) for _ in range(5))
        lr = 0.03 if kind == "sgd" else 1e-4
        torch.cuda.reset_peak_memory_stats()
        for _ in range(warmup):
            m.train_step(x1, x2, labels, LOSS_WEIGHT, lr=lr, optimizer=kind)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            losses = m.train_step(x1, x2, labels, LOSS_WEIGHT, lr=lr, optimizer=kind)
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        res[kind] = {"batch": B, "step_ms": dt * 1e3, "samples_per_s": B / dt, "steps_timed": steps,
                     "peak_allocated_gb": torch.cuda.max_memory_allocated() / 1e9,
                     "graph": m._engine._graph is not None, "losses_finite": bool(torch.isfinite(losses).all())}
        del m, x1, x2, labels, losses
        torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_optim_bench.json"))
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("optim_bench measures on a CUDA device; none is visible")
    out = {**card(), "hbm_reference_tbs": HBM_TBS, "launches": optimiser_launches(),
           "pretrain_step_b60": step_rates(a.steps, a.warmup)}
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
