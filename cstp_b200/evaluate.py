"""Video-level test evaluation: the loop of the reference's test.py:76-93 on the device.

test.py feeds one video at a time as a batch of its `n_clips` sliding windows through `model(inputs, None, o_type="test")`,
averages the logits over the clips and scores top-1 / top-5.  Here the clips of consecutive videos are packed into full
batches of one forward-only inference engine (eval BatchNorm couples no samples, so a clip's logits do not depend on its
batch), every batch is assembled by one clip-pipeline launch straight into the engine's static input, and the clip
averaging, top-k and hit counting run in two small kernels (csrc/video_eval.cu).  The host reads results back once.
"""
from __future__ import annotations

import math
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import engine as _engine_mod
from .data_process.clip_plan import FinetuneClipSampler
from .data_process.datasets import GpuVideoStore
from .data_process.gpu_clips import GpuClipPipeline

TOPK = 5


def shard(n: int, rank: int, world: int) -> range:
    """The contiguous range of videos rank `rank` of `world` scores: no padding, no duplicates."""
    return range(n * rank // world, n * (rank + 1) // world)


def batch_tables(counts: Sequence[int], capacity: int) -> np.ndarray:
    """Work lists of the accumulate / finalize kernels for every batch of `capacity` clips, the clips of videos 0, 1, ...
    (counts[v] clips each) packed in order: int32 [batches][2][capacity][3] with rows {slot = video, first row, clips in
    this batch} and {slot = video, clips of the video, video} of the videos whose last clip is in the batch; unused rows
    are zero (skipped)."""
    total = sum(counts)
    nb = math.ceil(total / capacity)
    tab = np.zeros((nb, 2, capacity, 3), dtype=np.int32)
    fill = np.zeros((nb, 2), dtype=np.int64)
    start = 0
    for v, n in enumerate(counts):
        end = start + n
        for b in range(start // capacity, (end - 1) // capacity + 1):
            lo, hi = max(start, b * capacity), min(end, (b + 1) * capacity)
            tab[b, 0, fill[b, 0]] = (v, lo - b * capacity, hi - lo)
            fill[b, 0] += 1
        b = (end - 1) // capacity
        tab[b, 1, fill[b, 1]] = (v, n, v)
        fill[b, 1] += 1
        start = end
    return tab


@torch.no_grad()
def test_videos(model, store: GpuVideoStore, total_frames: Sequence[int], labels: Sequence[int], *,
                sample_duration: int = 16, sample_size: int = 112, pb_rate: int = 4, capacity: int = 60, rank: int = 0,
                world: int = 1, keep_logits: bool = False, assemble: Optional[Callable] = None) -> dict:
    """Scores videos 0 .. len(total_frames) - 1 of `store` (the columns of testlist0X_nframe.txt: frame count and integer
    label) with the finetune model `model` (R21DBYOL(pretrain=False), DDP-wrapped or not) in eval semantics.

    Every video is cut into FinetuneClipSampler.plan_test windows; the clips of consecutive videos fill batches of
    `capacity` (a video may straddle batches).  With world > 1 this rank scores its contiguous shard and the hit counts
    are all-reduced over the default process group.  `assemble(plans, videos, out)` writes the clips of one batch into
    `out` (default: GpuClipPipeline.assemble_clips).

    Returns {"top1", "top5": accuracies over all ranks' videos, "hits": (top-1, top-5) hit counts, "videos", "clips":
    totals over all ranks, "predictions": int64 [shard videos][5] top-5 classes of this rank's videos, "logits": fp32
    [shard videos][num_classes] mean logits (keep_logits) or None}."""
    model = getattr(model, "module", model)
    ops = _engine_mod.ops
    T, S, C = int(sample_duration), int(sample_size), model.num_classes
    device = store.device
    mine = shard(len(total_frames), rank, world)
    sampler = FinetuneClipSampler(T, S, pb_rate)
    plans, owners = [], []
    for v in mine:
        vid = store[v]
        p = sampler.plan_test(int(total_frames[v]), vid.shape[2], vid.shape[1])
        plans.append(p)
        owners += [v] * len(p)
    clips = [c for p in plans for c in p]
    nv = len(mine)
    topk = torch.zeros(nv, TOPK, dtype=torch.int64, device=device)
    mean = torch.zeros(nv, C, dtype=torch.float32, device=device) if keep_logits else None
    counts = torch.tensor([0, 0, nv, len(clips)], dtype=torch.int64, device=device)   # top-1 hits, top-5 hits, videos, clips
    if clips:
        eng = model.inference_engine(capacity, T, S, S, device)
        model._repack_if_changed(eng)
        assemble = assemble or GpuClipPipeline(T, S, device).assemble_clips
        tables = torch.from_numpy(batch_tables([len(p) for p in plans], capacity)).to(device)
        y = torch.as_tensor([int(labels[v]) for v in mine], dtype=torch.int64).to(device)
        sums = torch.zeros(nv, C, dtype=torch.float32, device=device)
        for b in range(tables.shape[0]):
            rows = range(b * capacity, min(len(clips), (b + 1) * capacity))
            assemble([clips[i] for i in rows], [store[owners[i]] for i in rows], eng.x_static[:len(rows)])
            eng.run(len(rows))
            ops.video_accumulate(eng.logits, C, tables[b, 0], sums, rows=len(rows))
            ops.video_finalize(sums, tables[b, 1], topk, y, mean, counts[:2])
    if world > 1:
        torch.distributed.all_reduce(counts)
    counts = counts.cpu()
    hits1, hits5, videos, n_clips = (int(v) for v in counts)
    return {"top1": hits1 / max(videos, 1), "top5": hits5 / max(videos, 1), "hits": (hits1, hits5), "videos": videos,
            "clips": n_clips, "predictions": topk.cpu(), "logits": None if mean is None else mean.cpu()}
