"""Video-level test evaluation on one B200: cstp_b200.evaluate.test_videos (clips of consecutive videos packed into
batches of one inference engine) against the drop-in per-video loop of test.py:76-93 (model(clips, None, o_type="test"),
then mean and top-5 in torch), on a seeded synthetic test set resident in a GpuVideoStore.

    python tools/test_eval_bench.py [--baseline-root DIR] > test_eval_bench.json

--baseline-root DIR also runs the drop-in loop with the cstp_b200 package found in DIR (a checkout of another commit,
built), in a subprocess on the same GPU and the same seeded set, and checks its mean logits against this tree's.  Prints
one JSON line: card name and power limit, videos/s and clips/s of each path, engines built, device memory the inference
engines hold, and the batch-1 / batch-10 `o_type="test"` latency after a batch-60 finetune step (the protocol of
tools/finetune_bench.py)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

VIDEOS, SEED, CAPACITY = 200, 0, 60


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()[0]
    name, power = (s.strip() for s in q.split(","))
    return {"gpu": name, "power_limit": power}


def synthetic_set(n=VIDEOS):
    """Seeded frame counts log-uniform over [29, 1800] at 171x128, seeded pixels (drawn on the device) and labels."""
    from cstp_b200.data_process.datasets import GpuVideoStore
    g = torch.Generator().manual_seed(SEED)
    frames = torch.exp(torch.empty(n).uniform_(torch.log(torch.tensor(29.0)).item(), torch.log(torch.tensor(1800.0)).item(),
                                               generator=g)).round().int().tolist()
    frames[0], frames[1] = 29, 1800
    labels = torch.randint(0, 101, (n,), generator=g).tolist()
    store = GpuVideoStore()
    gd = torch.Generator(device="cuda").manual_seed(SEED)
    for v, f in enumerate(frames):
        store.put(v, torch.randint(0, 256, (f, 128, 171, 3), dtype=torch.uint8, device="cuda", generator=gd))
    return store, frames, labels


def model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    return R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda().eval()


def count_builds():
    from cstp_b200 import engine
    base = getattr(engine, "ProgramEngine", None) or engine.StepEngine     # every engine's constructor (older trees: StepEngine)
    built = []
    init = base.__init__

    def spy(self, B, *a, **k):
        built.append(B)
        init(self, B, *a, **k)
    base.__init__ = spy
    return built


def dropin_loop(m, store, frames, labels):
    """test.py:76-93 on the drop-in: one video per forward, mean over its clips and top-5 in torch."""
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    from cstp_b200.data_process.gpu_clips import GpuClipPipeline
    sampler, pipe = FinetuneClipSampler(16, 112, 4), GpuClipPipeline(16, 112)
    means, hits, clips = [], torch.zeros(2, dtype=torch.int64, device="cuda"), 0
    with torch.no_grad():
        for v, f in enumerate(frames):
            vid = store[v]
            plans = sampler.plan_test(f, vid.shape[2], vid.shape[1])
            x = pipe.assemble_clips(plans, [vid] * len(plans))
            mean = m(x, None, o_type="test").mean(0)
            top = torch.topk(mean, 5).indices
            hits[0] += top[0] == labels[v]
            hits[1] += (top == labels[v]).any()
            means.append(mean)
            clips += len(plans)
    means = torch.stack(means).cpu()
    return means, hits.cpu().tolist(), clips


def timed_pass(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def latency(m, x, iters=30, warm=5):
    """Eval-forward latency after a batch-60 finetune step (tools/finetune_bench.py)."""
    with torch.no_grad():
        for _ in range(warm):
            m(x, None, o_type="test")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            m(x, None, o_type="test")
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def dropin_arm(out_path):
    """The drop-in loop and the latency protocol with whichever cstp_b200 is first on sys.path."""
    built = count_builds()
    store, frames, labels = synthetic_set()
    m = model()
    before = torch.cuda.memory_allocated()
    t_first, (means, hits, clips) = timed_pass(lambda: dropin_loop(m, store, frames, labels))
    held = torch.cuda.memory_allocated() - before
    builds_first = len(built)
    t_second, _ = timed_pass(lambda: dropin_loop(m, store, frames, labels))
    res = {"first_pass_s": t_first, "second_pass_s": t_second, "videos_per_s": len(frames) / t_second,
           "clips_per_s": clips / t_second, "engines_built_first_pass": builds_first,
           "engines_built_second_pass": len(built) - builds_first, "engine_bytes": held, "hits": hits,
           "clips": clips}
    torch.save(means, out_path + ".means")
    del m
    torch.cuda.empty_cache()
    g = torch.Generator().manual_seed(0)
    x = (torch.rand(60, 3, 16, 112, 112, generator=g) * 2 - 1).cuda()
    y = torch.randint(0, 101, (60,), generator=g).cuda()
    m = model().train()
    m.finetune_step(x, y, lr=0.025, momentum=0.9, weight_decay=1e-3)
    m.eval()
    res["test_latency_b1_ms"] = latency(m, x[:1].contiguous())
    res["test_latency_b10_ms"] = latency(m, x[:10].contiguous())
    with open(out_path, "w") as f:
        json.dump(res, f)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline-root", default=None)
    ap.add_argument("--arm-out", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.arm_out:                         # subprocess: the drop-in arm with the package first on sys.path
        dropin_arm(a.arm_out)
        return
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    out = {**card(), "videos": VIDEOS, "capacity": CAPACITY}
    tmp = tempfile.mkdtemp()
    arms = {"dropin_this": root}
    if a.baseline_root:
        arms["dropin_baseline"] = os.path.abspath(a.baseline_root)
    for name, pkg in arms.items():
        path = os.path.join(tmp, name)
        env = dict(os.environ, PYTHONPATH=pkg)
        subprocess.run([sys.executable, os.path.abspath(__file__), "--arm-out", path], env=env, check=True, cwd=tmp)
        with open(path) as f:
            out[name] = json.load(f)
    means = {name: torch.load(os.path.join(tmp, name) + ".means") for name in arms}
    if "dropin_baseline" in means:
        out["dropin_mean_logits_equal_to_baseline"] = bool(torch.equal(means["dropin_this"], means["dropin_baseline"]))
    # ---- test_videos
    from cstp_b200.evaluate import test_videos
    built = count_builds()
    store, frames, labels = synthetic_set()
    m = model()
    before = torch.cuda.memory_allocated()
    t_first, r = timed_pass(lambda: test_videos(m, store, frames, labels, capacity=CAPACITY, keep_logits=True))
    held = torch.cuda.memory_allocated() - before
    times = [timed_pass(lambda: test_videos(m, store, frames, labels, capacity=CAPACITY))[0] for _ in range(3)]
    t = sorted(times)[1]
    out["test_videos"] = {"first_pass_s": t_first, "pass_s": times, "videos_per_s": r["videos"] / t,
                          "clips_per_s": r["clips"] / t, "engines_built": len(built), "hits": list(r["hits"]),
                          "clips": r["clips"], "top1": r["top1"], "top5": r["top5"],
                          "inference_engine_bytes": held}
    ref = means["dropin_this"]
    out["test_videos"]["mean_logits_max_abs_diff_vs_dropin_torch_mean"] = (r["logits"] - ref).abs().max().item()
    out["test_videos"]["top5_hits_equal_dropin"] = list(r["hits"]) == out["dropin_this"]["hits"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
