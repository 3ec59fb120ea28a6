"""Cost of monitoring a pretraining run on one B200: the collapse statistics inside the fused step, the statistics launch
on its own, and one RetrievalMonitor evaluation at UCF101 split-1 size.

    python tools/monitor_bench.py [--out profiles/r09_monitor_bench.json] [--rounds 5] [--steps 10]

1. The batch-60 pretraining step (R21DBYOL.train_step, 16x112x112 clips resident in HBM, the captured CUDA graph) with
   collapse_stats off and on, alternated in --rounds rounds on one model (each switch re-captures the step; two warm
   steps after a switch are not timed): mean step ms per round and arm, the within-arm spread, and the on - off
   difference of the arm medians.
2. cstp_repr_stats alone on that engine's buffers (4 blocks x 120 rows x 512 fp32, read three times per block from L2):
   mean us per launch over at least 1 s of back-to-back launches (CUDA events).
3. One RetrievalMonitor evaluation (features of 9,537 gallery and 3,783 query videos from the live batch-60 model, then
   the kNN search, k up to 50) on synthetic 171x128 videos: seeded log-normal lengths (median 160 frames, clipped to
   29 .. 1800), pixels taken from a pool of 32 seeded videos so that the store fits next to the training state; once
   from a GpuVideoStore and once from JPEG frames (a pool of 16 x 64 Pillow-encoded frames served by read_frames).
   Each source is warmed up on 64 videos first (engine build, graph capture), then timed once end to end.
The card's name, power limit and maximum SM clock are read in the same run.  Prints one JSON line and writes it to
--out."""
from __future__ import annotations

import argparse
import io
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LOSS_WEIGHT = (0.1, 1.0, 1.0, 1.0, 1.0)
B = 60
N_GALLERY, N_QUERY, N_CLASSES = 9537, 3783, 101
POOL, W, H = 32, 171, 128
MIN_TIMED_S = 1.0


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    name, power, clock = (s.strip() for s in q.split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def step_arms(m, rounds, steps):
    g = torch.Generator(device="cuda").manual_seed(2)
    x1 = torch.rand(B, 3, 16, 112, 112, device="cuda", generator=g) * 2 - 1
    x2 = torch.rand(B, 3, 16, 112, 112, device="cuda", generator=g) * 2 - 1
    labels = tuple(torch.randint(0, 5, (B,), device="cuda", generator=g) for _ in range(5))
    ms = {"off": [], "on": []}
    for _ in range(rounds):
        for arm in ("off", "on"):
            on = arm == "on"
            for _ in range(2):
                m.train_step(x1, x2, labels, LOSS_WEIGHT, lr=0.03, collapse_stats=on)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                losses = m.train_step(x1, x2, labels, LOSS_WEIGHT, lr=0.03, collapse_stats=on)
            torch.cuda.synchronize()
            ms[arm].append((time.perf_counter() - t0) / steps * 1e3)
    med = {a: statistics.median(v) for a, v in ms.items()}
    return {"batch": B, "steps_per_round": steps, "rounds": rounds, "step_ms": ms, "median_ms": med,
            "spread_ms": {a: max(v) - min(v) for a, v in ms.items()}, "on_minus_off_ms": med["on"] - med["off"],
            "samples_per_s_off": B / med["off"] * 1e3, "stats_last_step": m.step_stats().cpu().tolist(),
            "losses_finite": bool(torch.isfinite(losses).all())}


def stats_launch(m):
    from cstp_b200 import ops
    eng = m._engine
    out = torch.zeros(2, 5, device="cuda")

    def fn():
        ops.repr_stats(eng.feat, eng.proj_out, eng.pred, eng.tproj, eng.B, out)
    for _ in range(10):
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
    return {"launch_us": total / calls * 1e3, "launches_timed": calls, "rows_per_block": 2 * eng.B,
            "bytes_read_per_launch": 3 * 4 * 2 * eng.B * 512 * 4}


def synthetic_split(seed):
    g = np.random.default_rng(seed)
    n = N_GALLERY + N_QUERY
    frames = np.clip(np.round(np.exp(g.normal(np.log(160.0), 0.5, n))), 29, 1800).astype(int).tolist()
    labels = g.integers(0, N_CLASSES, n).tolist()
    return frames[:N_GALLERY], labels[:N_GALLERY], frames[N_GALLERY:], labels[N_GALLERY:]


def stores(gf, qf):
    from cstp_b200.data_process.datasets import GpuVideoStore
    gd = torch.Generator(device="cuda").manual_seed(7)
    pool = [torch.randint(0, 256, (1800, H, W, 3), dtype=torch.uint8, device="cuda", generator=gd) for _ in range(POOL)]
    out = []
    for base, frames in ((0, gf), (N_GALLERY, qf)):
        s = GpuVideoStore(capacity_bytes=1 << 60)          # the videos share the pool's storage
        for v, f in enumerate(frames):
            s.put(v, pool[(base + v) % POOL][:f])
        out.append(s)
    return out


def jpeg_readers():
    from PIL import Image
    g = np.random.default_rng(11)
    enc = []
    for _ in range(16):
        base = g.integers(0, 256, (H, W, 3), dtype=np.uint8)
        vid = []
        for k in range(64):
            b = io.BytesIO()
            Image.fromarray(np.roll(base, 3 * k, axis=1)).save(b, "JPEG", quality=90)
            vid.append(b.getvalue())
        enc.append(vid)

    def reader(base):
        def read_frames(video, numbers):
            e = enc[(base + video) % len(enc)]
            return [e[(f - 1) % 64] for f in numbers]
        return read_frames
    return reader(0), reader(N_GALLERY)


def evaluation(m, gf, gl, qf, ql):
    from cstp_b200.train import RetrievalMonitor
    from cstp_b200.evaluate import retrieve_videos, video_features
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    sampler = FinetuneClipSampler(16, 112, 4)
    clips = sum(len(sampler.plan_test(f, W, H)) for f in gf + qf)
    res = {"gallery_videos": len(gf), "query_videos": len(qf), "clips": clips, "mean_frames": float(np.mean(gf + qf))}
    gs, qs = stores(gf, qf)
    gr, qr = jpeg_readers()
    for name, (g_src, q_src) in (("store", (gs, qs)), ("jpeg", (gr, qr))):
        warm = RetrievalMonitor((g_src, gf[:64], gl[:64]), (q_src, qf[:64], ql[:64]))
        warm(m)
        mon = RetrievalMonitor((g_src, gf, gl), (q_src, qf, ql))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        rec = mon(m)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        res[name] = {"evaluation_s": dt, "videos_per_s": (len(gf) + len(qf)) / dt, "clips_per_s": clips / dt,
                     "recall": rec}
    g = video_features(m, gs, gf)
    q = video_features(m, qs, qf)
    retrieve_videos(q, ql, g, gl)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    retrieve_videos(q, ql, g, gl)
    res["knn_ms"] = (time.perf_counter() - t0) * 1e3
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_monitor_bench.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("monitor_bench measures on a CUDA device; none is visible")
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=True).cuda()
    out = {**card(), "pretrain_step_b60": step_arms(m, a.rounds, a.steps), "repr_stats_launch": stats_launch(m)}
    gf, gl, qf, ql = synthetic_split(3)
    out["retrieval_monitor_ucf101_split1"] = evaluation(m, gf, gl, qf, ql)
    out["peak_allocated_gb"] = torch.cuda.max_memory_allocated() / 1e9
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
