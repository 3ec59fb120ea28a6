"""Video-level test evaluation: the loop of the reference's test.py:76-93 on the device.

test.py feeds one video at a time as a batch of its `n_clips` sliding windows through `model(inputs, None, o_type="test")`,
averages the logits over the clips and scores top-1 / top-5.  Here the clips of consecutive videos are packed into full
batches of one forward-only inference engine (eval BatchNorm couples no samples, so a clip's logits do not depend on its
batch), every batch is assembled by one clip-pipeline launch straight into the engine's static input, and the clip
averaging, top-k and hit counting run in two small kernels (csrc/video_eval.cu).  The host reads results back once.

The same packing loop extracts per-video backbone features (video_features: the mean of the pooled 512-d feature in
front of the classification head), which retrieve_videos searches for nearest neighbours (csrc/retrieval.cu).

test_videos_jpeg / video_features_jpeg run the same loop from JPEG frames instead of a resident store: each batch
decodes only the frames its clips read, on the GPU, and the results are the store-fed call's bits.
"""
from __future__ import annotations

import itertools
import math
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import engine as _engine_mod
from .data_process.clip_plan import FinetuneClipSampler
from .data_process.datasets import GpuVideoStore, clip_frames
from .data_process.gpu_clips import GpuClipPipeline
from .data_process.jpeg import JpegSlabs

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


class _StoreFrames:
    """Test windows read from a resident GpuVideoStore."""

    def __init__(self, store: GpuVideoStore):
        self.store, self.device = store, store.device

    def frame_size(self, v: int):
        vid = self.store[v]
        return vid.shape[2], vid.shape[1]

    def batch(self, clips, owners):
        return clips, [self.store[v] for v in owners]

    def finish(self) -> None:
        pass


def batch_slabs(clips, owners):
    """What one packed batch decodes when it is fed from JPEG frames: the batch's clips grouped by video (the packing
    keeps a video's clips together), the distinct frames of each video's clips, and the clips remapped onto one slab per
    video (datasets.clip_frames).  Returns (videos, frame numbers per video, remapped clips, slab index per clip)."""
    videos, frames, remapped, slab = [], [], [], []
    for v, group in itertools.groupby(zip(owners, clips), key=lambda oc: oc[0]):
        fr, rc = clip_frames([c for _, c in group])
        slab += [len(videos)] * len(rc)
        videos.append(v)
        frames.append(fr)
        remapped += rc
    return videos, frames, remapped, slab


class _JpegFrames:
    """Test windows read from JPEG frames: per packed batch, only the frames its clips read are decoded, into a
    per-batch arena (jpeg.JpegSlabs); a rejected frame raises at the next batch or at the end of the call."""

    def __init__(self, read_frames, sizes, device):
        self.jpeg = JpegSlabs(read_frames, 1, sizes, device)
        self.device = self.jpeg.decoder.device

    def frame_size(self, v: int):
        return self.jpeg.frame_size(v)

    def batch(self, clips, owners):
        videos, frames, remapped, slab = batch_slabs(clips, owners)
        slabs = self.jpeg.decode(videos, frames)
        return remapped, [slabs[k] for k in slab]

    def finish(self) -> None:
        self.jpeg.check()


def _plan_clips(frames, total_frames: Sequence[int], videos: range, sampler: FinetuneClipSampler):
    """test.py's sliding windows of every video in `videos`: (per-video plans, flat clip list, owning video per clip)."""
    plans, owners = [], []
    for v in videos:
        w, h = frames.frame_size(v)
        p = sampler.plan_test(int(total_frames[v]), w, h)
        plans.append(p)
        owners += [v] * len(p)
    return plans, [c for p in plans for c in p], owners


def _pack_videos(model, frames, plans, clips, owners, *, T: int, S: int, capacity: int, source: str,
                 width: int, finalize: Callable, assemble: Optional[Callable] = None) -> None:
    """Runs the clips of consecutive videos through one inference engine in full batches of `capacity` and averages,
    per video, the first `width` columns of the engine's `source` rows ("logits" or "feat") in clip order.
    `finalize(sums, fin)` consumes the sums of the videos whose last clip is in the batch (cstp_video_finalize)."""
    ops = _engine_mod.ops
    device = frames.device
    eng = model.inference_engine(capacity, T, S, S, device)
    model._repack_if_changed(eng)
    assemble = assemble or GpuClipPipeline(T, S, device).assemble_clips
    tables = torch.from_numpy(batch_tables([len(p) for p in plans], capacity)).to(device)
    sums = torch.zeros(len(plans), width, dtype=torch.float32, device=device)
    for b in range(tables.shape[0]):
        rows = range(b * capacity, min(len(clips), (b + 1) * capacity))
        batch, videos = frames.batch([clips[i] for i in rows], [owners[i] for i in rows])
        assemble(batch, videos, eng.x_static[:len(rows)])
        eng.run(len(rows))
        ops.video_accumulate(getattr(eng, source), width, tables[b, 0], sums, rows=len(rows))
        finalize(sums, tables[b, 1])
    frames.finish()


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
    return _test_videos(model, _StoreFrames(store), total_frames, labels, sample_duration, sample_size, pb_rate, capacity,
                        rank, world, keep_logits, assemble)


@torch.no_grad()
def test_videos_jpeg(model, read_frames: Callable[[int, Sequence[int]], List[bytes]], total_frames: Sequence[int],
                     labels: Sequence[int], *, sizes: Optional[Sequence[Tuple[int, int]]] = None, device="cuda",
                     sample_duration: int = 16, sample_size: int = 112, pb_rate: int = 4, capacity: int = 60,
                     rank: int = 0, world: int = 1, keep_logits: bool = False) -> dict:
    """`test_videos` fed from JPEG frames instead of a store: the same windows, packing, results and bits.

    read_frames(video, frame_numbers) -> [bytes] returns the JPEG streams of those frames (1-based file numbers, as
    `FrameDirReader` reads them).  Each batch of `capacity` clips reads and decodes only the frames its clips use, in one
    call into a per-batch arena, so device memory holds one batch's frames, not the split's.  Frame sizes come from each
    video's first frame (read once) or from `sizes[video] = (w, h)`.  A rejected frame raises ValueError naming the video
    and the frame before the call returns."""
    return _test_videos(model, _JpegFrames(read_frames, sizes, device), total_frames, labels, sample_duration,
                        sample_size, pb_rate, capacity, rank, world, keep_logits, None)


def _test_videos(model, frames, total_frames, labels, sample_duration, sample_size, pb_rate, capacity, rank, world,
                 keep_logits, assemble) -> dict:
    model = getattr(model, "module", model)
    ops = _engine_mod.ops
    T, S, C = int(sample_duration), int(sample_size), model.num_classes
    device = frames.device
    mine = shard(len(total_frames), rank, world)
    plans, clips, owners = _plan_clips(frames, total_frames, mine, FinetuneClipSampler(T, S, pb_rate))
    nv = len(mine)
    topk = torch.zeros(nv, TOPK, dtype=torch.int64, device=device)
    mean = torch.zeros(nv, C, dtype=torch.float32, device=device) if keep_logits else None
    counts = torch.tensor([0, 0, nv, len(clips)], dtype=torch.int64, device=device)   # top-1 hits, top-5 hits, videos, clips
    if clips:
        y = torch.as_tensor([int(labels[v]) for v in mine], dtype=torch.int64).to(device)
        _pack_videos(model, frames, plans, clips, owners, T=T, S=S, capacity=capacity, source="logits", width=C,
                     finalize=lambda sums, fin: ops.video_finalize(sums, fin, topk, y, mean, counts[:2]),
                     assemble=assemble)
    if world > 1:
        torch.distributed.all_reduce(counts)
    counts = counts.cpu()
    hits1, hits5, videos, n_clips = (int(v) for v in counts)
    return {"top1": hits1 / max(videos, 1), "top5": hits5 / max(videos, 1), "hits": (hits1, hits5), "videos": videos,
            "clips": n_clips, "predictions": topk.cpu(), "logits": None if mean is None else mean.cpu()}


FEATURE_DIM = 512


@torch.no_grad()
def video_features(model, store: GpuVideoStore, total_frames: Sequence[int], *, sample_duration: int = 16,
                   sample_size: int = 112, pb_rate: int = 4, capacity: int = 60, rank: int = 0, world: int = 1,
                   assemble: Optional[Callable] = None) -> torch.Tensor:
    """Per-video backbone features of videos 0 .. len(total_frames) - 1 of `store`: the mean, over test.py's sliding
    windows (FinetuneClipSampler.plan_test), of the pooled 512-d feature in front of the classification head of the
    finetune model `model` (R21DBYOL(pretrain=False), DDP-wrapped or not) in eval semantics.  The clips are packed like
    test_videos'; a video's mean is its sequential fp32 sum in clip order divided by its clip count.

    `model` may also be a pretraining model (R21DBYOL(pretrain=True) that has run train_step): the features are then
    those of its live online network (engine_ft.FeatureEngine over the step engine's weights and BatchNorm running
    statistics), bit for bit the features of the finetune model loaded from a checkpoint of the same moment.  Nothing
    of the training state changes: no running statistic, no captured step, no optimiser state, no random generator.

    With world > 1 this rank extracts its contiguous shard and the shards are all-gathered over the default process
    group, so every rank returns all rows.  Returns fp32 [videos][512] on the store's device.  A split that does not fit
    in device memory is extracted chunk by chunk (one call per range of videos) and concatenated, or with
    video_features_jpeg."""
    return _video_features(model, _StoreFrames(store), total_frames, sample_duration, sample_size, pb_rate, capacity,
                           rank, world, assemble)


@torch.no_grad()
def video_features_jpeg(model, read_frames: Callable[[int, Sequence[int]], List[bytes]], total_frames: Sequence[int], *,
                        sizes: Optional[Sequence[Tuple[int, int]]] = None, device="cuda", sample_duration: int = 16,
                        sample_size: int = 112, pb_rate: int = 4, capacity: int = 60, rank: int = 0,
                        world: int = 1) -> torch.Tensor:
    """`video_features` fed from JPEG frames instead of a store, bit for bit the same features; `read_frames`, `sizes`
    and the per-batch decoding are those of test_videos_jpeg.  Device memory holds one batch's frames, so a split of
    any size is extracted in one call."""
    return _video_features(model, _JpegFrames(read_frames, sizes, device), total_frames, sample_duration, sample_size,
                           pb_rate, capacity, rank, world, None)


def _video_features(model, frames, total_frames, sample_duration, sample_size, pb_rate, capacity, rank, world,
                    assemble) -> torch.Tensor:
    model = getattr(model, "module", model)
    ops = _engine_mod.ops
    T, S = int(sample_duration), int(sample_size)
    device = frames.device
    n = len(total_frames)
    mine = shard(n, rank, world)
    plans, clips, owners = _plan_clips(frames, total_frames, mine, FinetuneClipSampler(T, S, pb_rate))
    feats = torch.zeros(len(mine), FEATURE_DIM, dtype=torch.float32, device=device)
    if clips:
        scratch = torch.zeros(len(mine), 1, dtype=torch.int64, device=device)      # finalize's top-k, unused
        _pack_videos(model, frames, plans, clips, owners, T=T, S=S, capacity=capacity, source="feat", width=FEATURE_DIM,
                     finalize=lambda sums, fin: ops.video_finalize(sums, fin, scratch, None, feats, None),
                     assemble=assemble)
    if world == 1:
        return feats
    most = -(-n // world)                           # shards differ in size by at most one: pad to the largest
    padded = torch.zeros(most, FEATURE_DIM, dtype=torch.float32, device=device)
    padded[:len(mine)] = feats
    parts = [torch.empty_like(padded) for _ in range(world)]
    torch.distributed.all_gather(parts, padded)
    return torch.cat([p[:len(shard(n, r, world))] for r, p in enumerate(parts)])


@torch.no_grad()
def retrieve_videos(query_feats: torch.Tensor, query_labels, gallery_feats: torch.Tensor, gallery_labels,
                    ks: Sequence[int] = (1, 5, 10, 20, 50), *, rank: int = 0, world: int = 1) -> dict:
    """Nearest-neighbour video retrieval (the VCOP / Pace protocol): every query video ranks the gallery videos by the
    cosine similarity of their features, and is a hit at k when one of its k nearest gallery videos has its label.

    query_feats fp32 [nq][d], gallery_feats fp32 [ng][d] (d % 4 == 0) on the device, labels int sequences or tensors
    with one entry per video; anything else raises ValueError.
    Both sets are L2-normalised (F.normalize) and searched by the fused similarity + top-k kernels of csrc/retrieval.cu
    in exact fp32: neighbours are ordered by similarity, then the lower gallery index, and do not depend on the tiling.
    With world > 1 this rank scores its contiguous shard of queries and the hit counts are all-reduced.

    Returns {"recall": {k: fraction of queries}, "hits": {k: count}, "queries": total over all ranks, "neighbours": int64
    [shard queries][max(ks)] gallery indices (-1 past the gallery), "similarity": fp32 [shard queries][max(ks)]}."""
    ops = _engine_mod.ops
    ks = [int(k) for k in ks]
    if not ks or min(ks) < 1 or max(ks) > 64:
        raise ValueError(f"retrieval cutoffs must lie in [1, 64], got {ks}")
    K = max(ks)
    for name, f in (("query", query_feats), ("gallery", gallery_feats)):
        if f.dtype != torch.float32 or f.dim() != 2:
            raise ValueError(f"{name} features must be a 2-D float32 tensor, got {f.dtype} {tuple(f.shape)}")
    if query_feats.device != gallery_feats.device:
        raise ValueError(f"query features on {query_feats.device}, gallery features on {gallery_feats.device}")
    device = query_feats.device
    mine = shard(query_feats.shape[0], rank, world)
    nq, ng, d = len(mine), gallery_feats.shape[0], gallery_feats.shape[1]
    if query_feats.shape[1] != d or d % 4 or ng < 1:
        raise ValueError(f"features must share a width that is a multiple of 4 and the gallery must not be empty: "
                         f"query {tuple(query_feats.shape)}, gallery {tuple(gallery_feats.shape)}")
    query_labels = torch.as_tensor(query_labels, dtype=torch.int64)
    gallery_labels = torch.as_tensor(gallery_labels, dtype=torch.int64)
    if query_labels.shape != (query_feats.shape[0],) or gallery_labels.shape != (ng,):
        raise ValueError(f"one label per video: {tuple(query_labels.shape)} labels for {query_feats.shape[0]} queries, "
                         f"{tuple(gallery_labels.shape)} for {ng} gallery videos")
    neighbours = torch.full((nq, K), -1, dtype=torch.int64, device=device)
    similarity = torch.full((nq, K), float("-inf"), dtype=torch.float32, device=device)
    counts = torch.zeros(len(ks) + 1, dtype=torch.int64, device=device)           # hits per cutoff, queries
    counts[-1] = nq
    if nq:
        q = torch.empty(nq, d, dtype=torch.float32, device=device)
        g = torch.empty(ng, d, dtype=torch.float32, device=device)
        ops.l2_normalize_rows(query_feats[mine.start:mine.stop].contiguous(), q)
        ops.l2_normalize_rows(gallery_feats.contiguous(), g)
        splits = ops.knn_splits(nq, ng)
        part_val = torch.empty(splits, nq, K, dtype=torch.float32, device=device)
        part_idx = torch.empty(splits, nq, K, dtype=torch.int32, device=device)
        ops.knn_partial(q, g, K, splits, part_val, part_idx)
        ql = query_labels[mine.start:mine.stop].to(device)
        gl = gallery_labels.to(device)
        cutoffs = torch.tensor(ks, dtype=torch.int32).to(device)
        ops.knn_merge(part_val, part_idx, neighbours, similarity, ql, gl, cutoffs, counts[:-1])
    if world > 1:
        torch.distributed.all_reduce(counts)
    counts = counts.cpu().tolist()
    queries = counts[-1]
    return {"recall": {k: counts[i] / max(queries, 1) for i, k in enumerate(ks)},
            "hits": {k: counts[i] for i, k in enumerate(ks)}, "queries": queries,
            "neighbours": neighbours.cpu(), "similarity": similarity.cpu()}
