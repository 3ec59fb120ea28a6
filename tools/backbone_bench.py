"""Cost of the standalone R2Plus1DNet (models.pace.r21d_byol, cstp_b200.engine_backbone) on one B200 at batch 60,
16x112x112 clips resident in HBM, with the projector (proj_flag=True, the BYOL online network):

    python tools/backbone_bench.py [--out profiles/r10_backbone_bench.json] [--iters 10] [--rounds 3]

1. train-mode forward + backward of one call (upstream gradients on feat and proj);
2. two calls + one backward (the BYOL online pattern);
3. both again with x.requires_grad (the stem input-gradient pass), and that kernel alone: mean us per launch over at
   least 1 s of back-to-back launches (CUDA events) on the engine's own d(raw), against its HBM floor (bytes it must
   move over 6.55 TB/s);
4. eval forward (capacity-60 engine) in clips/s, and of 1, 33 and 65 clips (capacity 1, 64 and 128 engines);
5. kernel launches per call (forward, backward, input gradient);
6. device memory one live arena holds (memory_allocated before / after building it) and the peak of a call;
7. the same module through stock PyTorch under bf16 autocast: oracle/cstp_oracle.r2plus1d_net (F.conv3d / F.batch_norm,
   cuDNN, channels_last_3d, cudnn.benchmark), items 1 and 2.
Times are host clocks around --iters iterations ending in a device synchronise, after two warm iterations, repeated in
--rounds rounds (the median and the spread are reported).  The card's name, power limit and maximum SM clock are read in
the same run.  Prints one JSON line and writes it to --out."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

B, T, S = 60, 16, 112
HBM_TBS = 6.55
MIN_TIMED_S = 1.0


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
    return {"median_ms": statistics.median(out), "spread_ms": max(out) - min(out), "rounds_ms": out}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_backbone_bench.json"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("backbone_bench needs a CUDA device")
    from cstp_b200 import ops
    from cstp_b200.models.pace.r21d_byol import R21DBYOL, R2Plus1DNet
    from oracle import cstp_oracle as O

    res = {"card": card(), "batch": B, "clip": [T, S, S], "proj_flag": True}
    torch.manual_seed(0)
    sd = {k[len("online_net."):]: v for k, v in R21DBYOL(pretrain=True).state_dict().items()
          if k.startswith("online_net.")}
    net = R2Plus1DNet(proj_flag=True)
    net.load_state_dict(sd)
    net.cuda().train()
    g = torch.Generator(device="cuda").manual_seed(2)
    x1 = torch.rand(B, 3, T, S, S, device="cuda", generator=g) * 2 - 1
    x2 = torch.rand(B, 3, T, S, S, device="cuda", generator=g) * 2 - 1
    uf = torch.randn(B, 512, device="cuda", generator=g)
    up = torch.randn(B, 512, device="cuda", generator=g)
    x1g, x2g = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)

    # ---- memory of one live arena (built by the first call), peak of a call
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    f, p = net(x1)
    torch.cuda.synchronize()
    m1 = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    torch.autograd.backward([f, p], [uf, up])
    torch.cuda.synchronize()
    res["first_arena_with_stores_bytes"] = m1 - m0
    res["peak_allocated_one_call_bytes"] = torch.cuda.max_memory_allocated()

    def one(x):
        def fn():
            f, p = net(x)
            torch.autograd.backward([f, p], [uf, up])
        return fn

    def two(xa, xb):
        def fn():
            fa, pa = net(xa)
            fb, pb = net(xb)
            torch.autograd.backward([fa, pa, fb, pb], [uf, up, uf, up])
        return fn

    # ---- launches per call
    n0 = ops.launch_count()
    f, p = net(x1g)
    n1 = ops.launch_count()
    torch.autograd.backward([f, p], [uf, up])
    torch.cuda.synchronize()
    n2 = ops.launch_count()
    res["launches"] = {"forward": n1 - n0, "backward_with_input_grad": n2 - n1, "input_grad": 1}
    two(x1, x2)()                               # second arena
    res["train_one_call_fwd_bwd"] = timed(one(x1), a.iters, a.rounds)
    res["train_two_calls_one_backward"] = timed(two(x1, x2), a.iters, a.rounds)
    res["train_one_call_fwd_bwd_input_grad"] = timed(one(x1g), a.iters, a.rounds)
    res["train_two_calls_one_backward_input_grad"] = timed(two(x1g, x2g), a.iters, a.rounds)
    torch.cuda.synchronize()
    res["peak_allocated_two_live_calls_bytes"] = torch.cuda.max_memory_allocated()

    # ---- the input-gradient kernel alone on the engine's d(raw)
    eng = next(e for k, pool in net._pools.items() if k[-1] == "grad" for e in pool)
    gbuf = eng._stem_holder["g"]
    w = eng.train.view("online_net.conv1.spatial_conv.weight")
    dx = torch.empty(B, 3, T, S, S, device="cuda")
    for _ in range(3):
        ops.stem_dgrad(gbuf, w, dx)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 0
    total_ms = 0.0
    while total_ms < MIN_TIMED_S * 1e3:
        ev0.record()
        for _ in range(50):
            ops.stem_dgrad(gbuf, w, dx)
        ev1.record()
        ev1.synchronize()
        total_ms += ev0.elapsed_time(ev1)
        n += 50
    us = total_ms / n * 1e3
    moved = gbuf.numel() * 2 + dx.numel() * 4
    flops = 2.0 * B * T * (S // 2) * (S // 2) * 83 * 3 * 49
    res["input_grad_kernel"] = {"us": us, "bytes": moved, "hbm_floor_us": moved / (HBM_TBS * 1e12) * 1e6,
                                "algorithmic_gflop": flops / 1e9, "tflops": flops / (us * 1e-6) / 1e12,
                                "note": "d(raw) read once and dx written once is the floor; the kernel re-reads the "
                                        "overlapping d(raw) rows of neighbouring tiles, mostly from L2"}

    # ---- eval forward at capacity 60
    net.eval()

    def ev():
        with torch.no_grad():
            net(x1)
    e = timed(ev, a.iters, a.rounds)
    e["clips_per_s"] = B / e["median_ms"] * 1e3
    res["eval_forward_capacity60"] = e
    n0 = ops.launch_count()
    ev()
    res["launches"]["eval_forward"] = ops.launch_count() - n0
    # batches below their capacity bucket (engine_ft.inference_capacity) run the bucket's whole program, as
    # InferenceEngine does: n = 33 and 65 run on the capacity-64 and capacity-128 engines
    xe = torch.cat([x1, x2[:5]])
    for n in (1, 33, 65):
        def evn(n=n):
            with torch.no_grad():
                net(xe[:n])
        e = timed(evn, a.iters, a.rounds)
        e["clips_per_s"] = n / e["median_ms"] * 1e3
        res[f"eval_forward_n{n}"] = e
    net.train()
    res["live_arenas"] = sum(len(pl) for pl in net._pools.values())
    del net, eng, gbuf, f, p
    torch.cuda.empty_cache()

    # ---- stock PyTorch under bf16 autocast
    torch.backends.cudnn.benchmark = True
    P = {"net." + k: v.cuda().requires_grad_("running" not in k and "num_batches" not in k) for k, v in sd.items()}
    xa = x1.contiguous(memory_format=torch.channels_last_3d)
    xb = x2.contiguous(memory_format=torch.channels_last_3d)

    def t_one():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            f, p = O.r2plus1d_net(xa, P, "net", {}, O.Tape(False), "a", proj=True)
        torch.autograd.backward([f.float(), p.float()], [uf, up])

    def t_two():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            fa, pa = O.r2plus1d_net(xa, P, "net", {}, O.Tape(False), "a", proj=True)
            fb, pb = O.r2plus1d_net(xb, P, "net", {}, O.Tape(False), "b", proj=True)
        torch.autograd.backward([fa.float(), pa.float(), fb.float(), pb.float()], [uf, up, uf, up])
    res["torch_bf16_autocast"] = {"train_one_call_fwd_bwd": timed(t_one, a.iters, a.rounds),
                                  "train_two_calls_one_backward": timed(t_two, a.iters, a.rounds)}
    line = json.dumps(res)
    print(line)
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        fh.write(line + "\n")


if __name__ == "__main__":
    main()
