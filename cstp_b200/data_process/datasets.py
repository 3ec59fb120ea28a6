"""Batch source of the pretraining loop on the GPU clip pipeline: what `get_data_loader` + `UcfRepreBYOLSpPre` /
`Kin400RepreLMDB` + `DistributedSampler` + `data_prefetcher` provide in the reference (utils.py:107-118,
data_process/datasets.py:806-948, 1253-1405, main_byol.py:33-49), with the pixel work on the device.

  * `GpuVideoStore`   decoded videos as uint8 [F][H][W][3] tensors in HBM, filled with decoded frames (`put`) or with
                      the JPEG bytes of pre-extracted frames, decoded on the GPU (`put_jpeg`, datasets.py:888).
  * `PretrainBatches` per epoch: the DistributedSampler's index order for this rank, one clip plan per sample drawn in
                      the reference's order, one `cstp_clip_assemble` launch per batch; yields
                      (clip_1, clip_2, (spa, tem, pb, rot_1, rot_2)) -- the argument order of `R21DBYOL.train_step`
                      and of `cstp_b200.train.pretrain_epochs` -- or, with `reference_format=True`, the DataLoader's own
                      `([clip_1, clip_2], [spa, tem, pb, [rot_1, rot_2]])` (main_byol.py:43-49).
  * `JpegPretrainBatches` the same batches, fed from JPEG frames read per batch and decoded on the GPU: no resident
                      store, so datasets of any size (Kinetics-400) can be pretrained.
  * `FinetuneBatches` / `JpegFinetuneBatches` the finetune and validation batches of `UcfFineTune` (datasets.py:951-1058)
                      for `cstp_b200.train.finetune_epochs`, from a store or from JPEG frames: (clips, labels).
"""
from __future__ import annotations

import math
from dataclasses import replace
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple

import torch

from .clip_plan import ClipPlan, FinetuneClipSampler, PretrainClipSampler, SamplePlan
from .gpu_clips import GpuClipPipeline, collate_labels
from .jpeg import GpuJpegDecoder, JpegSlabs, jpeg_size


class GpuVideoStore:
    """index -> CUDA uint8 tensor [F][H][W][3].  `capacity_bytes` bounds the resident set (least recently added videos
    are dropped first); a B200 holds ~2.7 M frames of 171x128 next to the training state."""

    def __init__(self, device="cuda", capacity_bytes: int = 100 << 30):
        self.device = torch.device(device)
        self.capacity = int(capacity_bytes)
        self.bytes = 0
        self._vids: Dict[int, torch.Tensor] = {}
        self._jpeg = None

    def put(self, idx: int, frames) -> None:
        t = torch.as_tensor(frames)
        if t.dtype != torch.uint8 or t.dim() != 4 or t.shape[3] != 3:
            raise ValueError("frames must be uint8 [F][H][W][3]")
        self._insert(idx, t.to(self.device, non_blocking=True).contiguous())

    def put_jpeg(self, idx: int, streams: Sequence[bytes]) -> None:
        """Stores video idx from the JPEG bytes of its frames (in frame order), decoded on the GPU byte for byte as
        Pillow decodes them.  Every frame must have the first frame's size.  Raises ValueError naming the first
        rejected frame (this waits for the decode)."""
        if not streams:
            raise ValueError("a video needs at least one frame")
        w, h = jpeg_size(streams[0])
        t = torch.empty((len(streams), h, w, 3), dtype=torch.uint8, device=self.device)
        if self._jpeg is None:
            self._jpeg = GpuJpegDecoder(self.device)
        status = self._jpeg.decode(streams, [(w, h)] * len(streams), list(t))
        GpuJpegDecoder.check(status, [f"video {idx} frame index {k}" for k in range(len(streams))])
        self._insert(idx, t)

    def _insert(self, idx: int, t: torch.Tensor) -> None:
        if idx in self._vids:
            self.bytes -= self._vids.pop(idx).numel()
        while self._vids and self.bytes + t.numel() > self.capacity:
            self.bytes -= self._vids.pop(next(iter(self._vids))).numel()
        self._vids[idx] = t
        self.bytes += t.numel()

    def __contains__(self, idx: int) -> bool:
        return idx in self._vids

    def __getitem__(self, idx: int) -> torch.Tensor:
        return self._vids[idx]

    def __len__(self) -> int:
        return len(self._vids)


def distributed_indices(n: int, epoch: int, rank: int = 0, world: int = 1, seed: int = 0, shuffle: bool = True) -> List[int]:
    """torch.utils.data.DistributedSampler's order for this rank (shuffle, drop_last=False): what utils.py:109-110 builds
    and main_byol.py:261 re-seeds with `set_epoch`."""
    if shuffle:
        g = torch.Generator()
        g.manual_seed(seed + epoch)
        idx = torch.randperm(n, generator=g).tolist()
    else:
        idx = list(range(n))
    total = math.ceil(n / world) * world
    pad = total - len(idx)
    if pad > 0:
        idx += (idx * math.ceil(pad / len(idx)))[:pad]
    return idx[rank:total:world]


class _EpochBatches:
    """The batch loop the batch sources share: per epoch, this rank's DistributedSampler order cut into batches (the last
    one partial unless drop_last), each built by `_batch(ids, slot)` into one of two alternating output slots, so that
    batch b + 1 is assembled while the step on batch b runs."""

    def _configure_epochs(self, device, total_frames, batch_size, sample_duration, sample_size, rank, world, seed,
                          shuffle, drop_last):
        self.device, self.total_frames = torch.device(device), list(total_frames)
        self.batch_size = int(batch_size)
        self.pipe = GpuClipPipeline(sample_duration, sample_size, self.device)
        self.rank, self.world, self.seed, self.shuffle, self.drop_last = rank, world, seed, shuffle, drop_last
        self._out = [None, None]

    def __call__(self, epoch: int) -> Iterator:
        order = distributed_indices(len(self.total_frames), epoch, self.rank, self.world, self.seed, self.shuffle)
        nb = len(order) // self.batch_size if self.drop_last else math.ceil(len(order) / self.batch_size)
        for b in range(nb):
            yield self._batch(order[b * self.batch_size:(b + 1) * self.batch_size], b & 1)


class PretrainBatches(_EpochBatches):
    """`batches(epoch)` for `cstp_b200.train.pretrain_epochs`.

    total_frames[i] is the annotated frame count of video i (the third column of trainlist0X_nframe.txt,
    datasets.py:826-827); the store must hold at least that many frames (+ frame 0 unused for the 1-based UCF layout is
    NOT needed: store[i][k] is file number k + 1)."""

    def __init__(self, store: GpuVideoStore, total_frames: Sequence[int], batch_size: int, variant: str = "ucf",
                 sample_duration: int = 16, sample_size: int = 112, rank: int = 0, world: int = 1, seed: int = 0,
                 shuffle: bool = True, drop_last: bool = True, reference_format: bool = False):
        self.store = store
        self._configure(store.device, total_frames, batch_size, variant, sample_duration, sample_size, rank, world, seed,
                        shuffle, drop_last, reference_format)

    def _configure(self, device, total_frames, batch_size, variant, sample_duration, sample_size, rank, world, seed,
                   shuffle, drop_last, reference_format):
        self._configure_epochs(device, total_frames, batch_size, sample_duration, sample_size, rank, world, seed, shuffle,
                               drop_last)
        self.sampler = PretrainClipSampler(sample_duration, sample_size, variant)
        self.reference_format = reference_format

    def _videos(self, ids: Sequence[int]):
        """One batch's plans, drawn in the order of `ids`, and the frame tensors they read."""
        plans, vids = [], []
        for i in ids:
            vid = self.store[i]
            plans.append(self.sampler.plan(self.total_frames[i], vid.shape[2], vid.shape[1]))
            vids.append(vid)
        return plans, vids

    def _batch(self, ids: Sequence[int], slot: int):
        plans, vids = self._videos(ids)
        if self._out[slot] is not None and self._out[slot][0].shape[0] != len(ids):
            self._out[slot] = None
        self._out[slot] = self.pipe.assemble(plans, vids, self._out[slot])
        x1, x2 = self._out[slot]
        spa, tem, pb, (r1, r2) = collate_labels(plans, device=self.device)
        if self.reference_format:
            return [x1, x2], [spa, tem, pb, [r1, r2]]
        return x1, x2, (spa, tem, pb, r1, r2)


class FinetuneBatches(_EpochBatches):
    """`train_batches` / `val_batches` for `cstp_b200.train.finetune_epochs`: `batches(epoch)` yields (clips fp32
    [B][3][T][S][S], labels int64 [B]) on the store's device, the batches `UcfFineTune` (datasets.py:951-1058) under
    get_transforms('img') or ('img_val') hands main_ft_mp.py:196-214 / 255-289 through a DistributedSampler.

    Per epoch: this rank's `distributed_indices` order (seeded by seed + epoch).  Per sample: one
    FinetuneClipSampler.plan_train (split "train": random sized crop, colour jitter) or plan_val (split "val": scale and
    centre crop) draw, in the order the samples appear in the batch, as `UcfFineTune.__getitem__` draws them when one
    process calls it in that order.  Per batch: one `cstp_clip_assemble` launch into one of two alternating buffers.

    total_frames[i] is the frame count of video i (the third column of the *_nframe.txt lists) and labels[i] its class
    index (the second column); store[i][k] is frame file k + 1.  shuffle / drop_last default to True / True for "train",
    so every step runs at the batch size the fused step is bound to, and to False / False for "val", whose last partial
    batch runs on an inference engine.  These defaults are this package's choice; they are not taken from the
    reference's loader construction (`utils.get_dataloader`)."""

    def __init__(self, store: GpuVideoStore, total_frames: Sequence[int], labels: Sequence[int], batch_size: int,
                 split: str = "train", sample_duration: int = 16, sample_size: int = 112, pb_rate: int = 4, rank: int = 0,
                 world: int = 1, seed: int = 0, shuffle: Optional[bool] = None, drop_last: Optional[bool] = None):
        self.store = store
        self._configure(store.device, total_frames, labels, batch_size, split, sample_duration, sample_size, pb_rate,
                        rank, world, seed, shuffle, drop_last)

    def _configure(self, device, total_frames, labels, batch_size, split, sample_duration, sample_size, pb_rate, rank,
                   world, seed, shuffle, drop_last):
        if split not in ("train", "val"):
            raise ValueError(f"split must be 'train' or 'val', got {split!r}")
        if len(labels) != len(total_frames):
            raise ValueError(f"one label per video: {len(labels)} labels for {len(total_frames)} videos")
        train = split == "train"
        self._configure_epochs(device, total_frames, batch_size, sample_duration, sample_size, rank, world, seed,
                               train if shuffle is None else shuffle, train if drop_last is None else drop_last)
        self.split, self.labels = split, [int(y) for y in labels]
        sampler = FinetuneClipSampler(sample_duration, sample_size, pb_rate)
        self.draw = sampler.plan_train if train else sampler.plan_val

    def _videos(self, ids: Sequence[int]):
        """One batch's clip plans, drawn in the order of `ids`, and the frame tensors they read."""
        plans, vids = [], []
        for i in ids:
            vid = self.store[i]
            plans.append(self.draw(self.total_frames[i], vid.shape[2], vid.shape[1]))
            vids.append(vid)
        return plans, vids

    def _batch(self, ids: Sequence[int], slot: int):
        plans, vids = self._videos(ids)
        if self._out[slot] is not None and self._out[slot].shape[0] != len(ids):
            self._out[slot] = None
        self._out[slot] = self.pipe.assemble_clips(plans, vids, self._out[slot])
        labels = torch.tensor([self.labels[i] for i in ids], dtype=torch.int64).to(self.device, non_blocking=True)
        return self._out[slot], labels


def distinct_frames(plan: SamplePlan) -> Tuple[List[int], SamplePlan]:
    """The frame numbers one sample reads over both views, sorted and without repeats (the Kinetics variant's second
    view re-reads the first view's frames), and the plan with its frame numbers remapped onto a slab holding exactly
    those frames: slab[k] is frame frames[k], read by the pipeline as frame number `plan.frame_base + k`."""
    frames = sorted({f for v in plan.views for f in v.frames})
    pos = {f: k + plan.frame_base for k, f in enumerate(frames)}
    views = tuple(replace(v, frames=[pos[f] for f in v.frames]) for v in plan.views)
    return frames, replace(plan, views=views)


def clip_frames(clips: Sequence[ClipPlan]) -> Tuple[List[int], List[ClipPlan]]:
    """`distinct_frames` for one-view clips of one video: the frame numbers the clips read, sorted and without repeats
    (a short video wraps around and reads a frame twice; consecutive test windows share a frame), and the clips remapped
    onto a slab holding exactly those frames: slab[k] is frame frames[k], read as frame number `frame_base + k`."""
    frames = sorted({f for c in clips for f in c.view.frames})
    base = clips[0].frame_base
    pos = {f: k + base for k, f in enumerate(frames)}
    return frames, [replace(c, view=replace(c.view, frames=[pos[f] for f in c.view.frames])) for c in clips]


class _JpegFed:
    """What the JPEG-fed batch sources add to their store-fed base: `_plan(ids)` returns the batch's plans, remapped onto
    per-sample slabs, and the frames each sample reads; `_videos` decodes those frames through `self.jpeg`
    (jpeg.JpegSlabs), and a rejected frame raises when the next batch, or the end of the epoch, is requested."""

    def frame_size(self, video: int) -> Tuple[int, int]:
        return self.jpeg.frame_size(video)

    def _videos(self, ids: Sequence[int]):
        self.jpeg.check()
        plans, frames = self._plan(ids)
        return plans, self.jpeg.decode(ids, frames)

    def __call__(self, epoch: int) -> Iterator:
        self.jpeg.check()
        yield from super().__call__(epoch)
        self.jpeg.check()


class JpegPretrainBatches(_JpegFed, PretrainBatches):
    """`PretrainBatches` fed from JPEG frames instead of a store: same arguments, iteration, random draws and outputs.

    read_frames(video, frame_numbers) -> [bytes] returns the JPEG streams of those frames of a video (frame numbers as
    the plans use them: 1-based file numbers for "ucf", 0-based list indices for "kinetics"); `FrameDirReader` reads
    frame directories.  Per batch, each sample's distinct frames are read, uploaded once and decoded in one call into a
    per-batch arena (one [n][H][W][3] slab per sample) on the current stream, then assembled as `PretrainBatches` does.
    Frame sizes come from the first frame of each video (cached), or from `sizes[video] = (w, h)` when given.

    Decode errors are checked without stalling the stream: a rejected frame of batch b raises ValueError, naming the
    video and the frame, when batch b + 1 (or the end of the epoch) is requested.  By then the consumer may already have
    run a step on batch b, whose rejected frames' pixels are unspecified."""

    def __init__(self, read_frames: Callable[[int, Sequence[int]], List[bytes]], total_frames: Sequence[int],
                 batch_size: int, variant: str = "ucf", sample_duration: int = 16, sample_size: int = 112, rank: int = 0,
                 world: int = 1, seed: int = 0, shuffle: bool = True, drop_last: bool = True,
                 reference_format: bool = False, sizes: Optional[Sequence[Tuple[int, int]]] = None, device="cuda"):
        self._configure(device, total_frames, batch_size, variant, sample_duration, sample_size, rank, world, seed,
                        shuffle, drop_last, reference_format)
        self.jpeg = JpegSlabs(read_frames, 1 if variant == "ucf" else 0, sizes, self.device)

    def _plan(self, ids: Sequence[int]):
        """The batch's plans (remapped onto per-sample slabs) and each sample's distinct frame numbers; the sampler is
        called exactly as `PretrainBatches` calls it."""
        plans, frames = [], []
        for i in ids:
            w, h = self.frame_size(i)
            fr, plan = distinct_frames(self.sampler.plan(self.total_frames[i], w, h))
            plans.append(plan)
            frames.append(fr)
        return plans, frames


class JpegFinetuneBatches(_JpegFed, FinetuneBatches):
    """`FinetuneBatches` fed from JPEG frames instead of a store: same arguments, iteration, random draws and outputs,
    with `read_frames`, `sizes` and the decode-error contract of `JpegPretrainBatches` (frame numbers are 1-based file
    numbers).  Per batch, each clip's distinct frames are read and decoded in one call into per-sample slabs."""

    def __init__(self, read_frames: Callable[[int, Sequence[int]], List[bytes]], total_frames: Sequence[int],
                 labels: Sequence[int], batch_size: int, split: str = "train", sample_duration: int = 16,
                 sample_size: int = 112, pb_rate: int = 4, rank: int = 0, world: int = 1, seed: int = 0,
                 shuffle: Optional[bool] = None, drop_last: Optional[bool] = None,
                 sizes: Optional[Sequence[Tuple[int, int]]] = None, device="cuda"):
        self._configure(device, total_frames, labels, batch_size, split, sample_duration, sample_size, pb_rate, rank,
                        world, seed, shuffle, drop_last)
        self.jpeg = JpegSlabs(read_frames, 1, sizes, self.device)

    def _plan(self, ids: Sequence[int]):
        """The batch's clip plans (remapped onto per-sample slabs) and each clip's distinct frame numbers; the sampler
        is called exactly as `FinetuneBatches` calls it."""
        plans, frames = [], []
        for i in ids:
            w, h = self.frame_size(i)
            fr, (plan,) = clip_frames([self.draw(self.total_frames[i], w, h)])
            plans.append(plan)
            frames.append(fr)
        return plans, frames
