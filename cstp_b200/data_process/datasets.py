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
"""
from __future__ import annotations

import math
from dataclasses import replace
from typing import Callable, Dict, Iterator, List, Optional, Sequence, Tuple

import torch

from .clip_plan import PretrainClipSampler, SamplePlan
from .gpu_clips import GpuClipPipeline, collate_labels
from .jpeg import GpuJpegDecoder, jpeg_size, raise_for_status


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


class PretrainBatches:
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
        self.device, self.total_frames = torch.device(device), list(total_frames)
        self.batch_size = int(batch_size)
        self.sampler = PretrainClipSampler(sample_duration, sample_size, variant)
        self.pipe = GpuClipPipeline(sample_duration, sample_size, self.device)
        self.rank, self.world, self.seed, self.shuffle, self.drop_last = rank, world, seed, shuffle, drop_last
        self.reference_format = reference_format
        self._out = [None, None]                  # two output buffer pairs: batch i+1 is assembled while step i runs

    def _videos(self, ids: Sequence[int]):
        """One batch's plans, drawn in the order of `ids`, and the frame tensors they read."""
        plans, vids = [], []
        for i in ids:
            vid = self.store[i]
            plans.append(self.sampler.plan(self.total_frames[i], vid.shape[2], vid.shape[1]))
            vids.append(vid)
        return plans, vids

    def __call__(self, epoch: int) -> Iterator:
        order = distributed_indices(len(self.total_frames), epoch, self.rank, self.world, self.seed, self.shuffle)
        nb = len(order) // self.batch_size if self.drop_last else math.ceil(len(order) / self.batch_size)
        for b in range(nb):
            ids = order[b * self.batch_size:(b + 1) * self.batch_size]
            plans, vids = self._videos(ids)
            slot = b & 1
            if self._out[slot] is not None and self._out[slot][0].shape[0] != len(ids):
                self._out[slot] = None
            self._out[slot] = self.pipe.assemble(plans, vids, self._out[slot])
            x1, x2 = self._out[slot]
            spa, tem, pb, (r1, r2) = collate_labels(plans, device=self.device)
            if self.reference_format:
                yield [x1, x2], [spa, tem, pb, [r1, r2]]
            else:
                yield x1, x2, (spa, tem, pb, r1, r2)


def distinct_frames(plan: SamplePlan) -> Tuple[List[int], SamplePlan]:
    """The frame numbers one sample reads over both views, sorted and without repeats (the Kinetics variant's second
    view re-reads the first view's frames), and the plan with its frame numbers remapped onto a slab holding exactly
    those frames: slab[k] is frame frames[k], read by the pipeline as frame number `plan.frame_base + k`."""
    frames = sorted({f for v in plan.views for f in v.frames})
    pos = {f: k + plan.frame_base for k, f in enumerate(frames)}
    views = tuple(replace(v, frames=[pos[f] for f in v.frames]) for v in plan.views)
    return frames, replace(plan, views=views)


class JpegPretrainBatches(PretrainBatches):
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
        self.read_frames = read_frames
        self._configure(device, total_frames, batch_size, variant, sample_duration, sample_size, rank, world, seed,
                        shuffle, drop_last, reference_format)
        self.decoder = GpuJpegDecoder(self.device)
        self._sizes: Dict[int, Tuple[int, int]] = {i: tuple(s) for i, s in enumerate(sizes)} if sizes is not None else {}
        self._pending = None                       # (pinned status, event, frame names) of the last decode

    def frame_size(self, video: int) -> Tuple[int, int]:
        if video not in self._sizes:
            first = 1 if self.sampler.variant == "ucf" else 0
            self._sizes[video] = jpeg_size(self.read_frames(video, [first])[0])
        return self._sizes[video]

    def _check_pending(self) -> None:
        if self._pending is not None:
            host, ev, names = self._pending
            self._pending = None
            ev.synchronize()
            raise_for_status(host.numpy(), names)

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

    def _videos(self, ids: Sequence[int]):
        self._check_pending()
        plans, frames = self._plan(ids)
        sizes = [self.frame_size(i) for i in ids]
        arena = torch.empty(sum(len(fr) * w * h * 3 for fr, (w, h) in zip(frames, sizes)), dtype=torch.uint8,
                            device=self.device)
        streams, exp, outs, names, vids = [], [], [], [], []
        off = 0
        for i, fr, (w, h) in zip(ids, frames, sizes):
            slab = arena[off:off + len(fr) * h * w * 3].view(len(fr), h, w, 3)
            off += slab.numel()
            data = self.read_frames(i, fr)
            if len(data) != len(fr):
                raise ValueError(f"read_frames returned {len(data)} streams for {len(fr)} frames of video {i}")
            streams += data
            exp += [(w, h)] * len(fr)
            outs += list(slab)
            names += [f"video {i} frame {f}" for f in fr]
            vids.append(slab)
        status = self.decoder.decode(streams, exp, outs)
        host = torch.empty(len(streams), dtype=torch.int32).pin_memory()
        host.copy_(status, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pending = (host, ev, names)
        return plans, vids

    def __call__(self, epoch: int) -> Iterator:
        self._check_pending()
        yield from super().__call__(epoch)
        self._check_pending()
