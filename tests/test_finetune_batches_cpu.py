"""Host logic of the finetune / validation batch sources and of the JPEG-fed evaluation: batch composition against a
restatement (torch's DistributedSampler order, FinetuneClipSampler called in that order), the one-view frame remap,
the frame-size cache, the read_frames count check, and which frames each packed evaluation batch decodes."""
import random

import numpy as np
import pytest
import torch
from torch.utils.data import DistributedSampler

from cstp_b200.data_process.clip_plan import FinetuneClipSampler
from cstp_b200.data_process.datasets import FinetuneBatches, JpegFinetuneBatches, clip_frames
from cstp_b200.evaluate import batch_slabs, batch_tables

SIZES = [(171, 128), (161, 121), (173, 131), (340, 256), (171, 128), (149, 113), (171, 128)]
COUNTS = [40, 157, 33, 64, 20, 90, 61]
LABELS = [100 - 7 * i for i in range(len(COUNTS))]            # distinct: a batch's labels name its videos


class _ShapeStore:
    """Stand-in for GpuVideoStore that only answers shapes (what FinetuneBatches reads to plan a batch)."""
    device = torch.device("cpu")

    def __getitem__(self, i):
        w, h = SIZES[i]
        return torch.empty((1, 1, 1, 3), dtype=torch.uint8).expand(COUNTS[i], h, w, 3)


class _RecordingPipe:
    """Records the plans of every assemble_clips launch instead of running the kernel."""

    def __init__(self):
        self.plans = []

    def assemble_clips(self, plans, videos, out=None):
        assert len(videos) == len(plans)
        self.plans.append(list(plans))
        return torch.zeros(len(plans))


def _seed(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


def _restated(split, epoch, rank, world, seed, batch_size):
    """What one process of the reference draws: DistributedSampler(shuffle, seed).set_epoch(epoch) for this rank, cut
    into batches, UcfFineTune's clip draws for every sample in that order."""
    train = split == "train"
    ds = DistributedSampler(range(len(COUNTS)), num_replicas=world, rank=rank, shuffle=train, seed=seed)
    ds.set_epoch(epoch)
    order = list(ds)
    batches = [order[k:k + batch_size] for k in range(0, len(order), batch_size)]
    if train and len(batches[-1]) < batch_size:
        batches.pop()
    sampler = FinetuneClipSampler(16, 112, 4)
    draw = sampler.plan_train if train else sampler.plan_val
    return [([LABELS[i] for i in ids], [draw(COUNTS[i], *SIZES[i]) for i in ids]) for ids in batches]


@pytest.mark.parametrize("split", ["train", "val"])
@pytest.mark.parametrize("rank,world", [(0, 1), (1, 2)])
def test_batches_follow_the_distributed_order_and_the_reference_draws(split, rank, world):
    src = FinetuneBatches(_ShapeStore(), COUNTS, LABELS, 3, split=split, rank=rank, world=world, seed=4)
    src.pipe = _RecordingPipe()
    assert (src.shuffle, src.drop_last) == ((True, True) if split == "train" else (False, False))
    partial = False
    for epoch in range(2):
        _seed(20 + epoch)
        want = _restated(split, epoch, rank, world, 4, 3)
        after_ref = (random.random(), np.random.rand(), torch.rand(1).item())
        _seed(20 + epoch)
        src.pipe.plans.clear()
        got = [labels.tolist() for _, labels in src(epoch)]
        after = (random.random(), np.random.rand(), torch.rand(1).item())
        assert after == after_ref                                   # the same draws, and no others
        assert got == [labels for labels, _ in want]
        assert src.pipe.plans == [plans for _, plans in want]
        partial |= len(got[-1]) < 3
    assert partial == (split == "val")                            # 7 videos (4 per rank at world 2): val ends partial


def test_jpeg_source_plans_like_the_store_source():
    reads = []

    def read_frames(video, frames):
        reads.append((video, list(frames)))
        return [b""] * len(frames)

    for split in ("train", "val"):
        ref = FinetuneBatches(_ShapeStore(), COUNTS, LABELS, 4, split=split)
        src = JpegFinetuneBatches(read_frames, COUNTS, LABELS, 4, split=split, sizes=SIZES, device="cpu")
        ids = [4, 1, 6, 2]
        for trial in range(3):
            _seed(trial)
            want, _ = ref._videos(ids)
            state_ref = (random.random(), np.random.rand(), torch.rand(1).item())
            _seed(trial)
            plans, frames = src._plan(ids)
            assert (random.random(), np.random.rand(), torch.rand(1).item()) == state_ref
            for p, w, fr in zip(plans, want, frames):
                assert fr == sorted(set(w.view.frames))
                assert [fr[k - 1] for k in p.view.frames] == w.view.frames
                assert (p.view.box, p.view.resize, p.view.base, p.view.jitter, p.frame_base) == \
                    (w.view.box, w.view.resize, w.view.base, w.view.jitter, w.frame_base)
    assert not reads                                                # sizes given: no frame read to plan


def test_clip_frames_deduplicates_wrapped_and_shared_frames():
    _seed(1)
    sampler = FinetuneClipSampler(16, 112, 4)
    short = sampler.plan_val(20, 171, 128)                          # 20 frames < one window: wraps to frame 1
    assert short.view.frames[:6] == [1, 5, 9, 13, 17, 1]
    frames, (remapped,) = clip_frames([short])
    assert frames == [1, 5, 9, 13, 17]
    assert remapped.view.frames[:6] == [1, 2, 3, 4, 5, 1] and short.view.frames[:6] == [1, 5, 9, 13, 17, 1]
    assert [frames[k - 1] for k in remapped.view.frames] == short.view.frames
    windows = sampler.plan_test(130, 171, 128)                      # windows at 1, 61 and the last one, 70
    frames, remapped = clip_frames(windows)
    assert frames == sorted({f for w in windows for f in w.view.frames}) and len(frames) < 3 * 16
    for w, r in zip(windows, remapped):
        assert [frames[k - 1] for k in r.view.frames] == w.view.frames
        assert (r.view.box, r.view.resize) == (w.view.box, w.view.resize)


def test_frame_size_reads_the_first_frame_once():
    from tests import jpeg_cases as J
    b = J.pil_encode(J.content("video", 45, 31), "420", quality=80)
    calls = []

    def read_frames(video, frames):
        calls.append((video, list(frames)))
        return [b] * len(frames)
    src = JpegFinetuneBatches(read_frames, [20, 30], [0, 1], 1, device="cpu")
    assert src.frame_size(1) == (45, 31) and src.frame_size(1) == (45, 31) and src.frame_size(0) == (45, 31)
    assert calls == [(1, [1]), (0, [1])]


def test_read_frames_returning_the_wrong_count_raises():
    def short_read(video, frames):
        return [b""] * (len(frames) - 1)
    src = JpegFinetuneBatches(short_read, COUNTS, LABELS, 2, split="val", sizes=SIZES, device="cpu")
    with pytest.raises(ValueError, match=r"read_frames returned \d+ streams for \d+ frames of video 0"):
        next(iter(src(0)))


def test_labels_and_split_are_checked():
    with pytest.raises(ValueError, match="one label per video"):
        FinetuneBatches(_ShapeStore(), COUNTS, LABELS[:-1], 2)
    with pytest.raises(ValueError, match="split"):
        FinetuneBatches(_ShapeStore(), COUNTS, LABELS, 2, split="test")


@pytest.mark.parametrize("capacity", [1, 3, 7, 60])
def test_evaluation_batches_decode_only_the_frames_their_clips_read(capacity):
    sampler = FinetuneClipSampler(16, 112, 4)
    frames_of = [29, 95, 200, 61, 130, 45, 64, 250]                 # 29 and 45: shorter than one window
    clips, owners, plans = [], [], []
    for v, n in enumerate(frames_of):
        p = sampler.plan_test(n, 171, 128)
        plans.append(p)
        clips += p
        owners += [v] * len(p)
    decoded = {}
    for b in range(batch_tables([len(p) for p in plans], capacity).shape[0]):
        rows = range(b * capacity, min(len(clips), (b + 1) * capacity))
        bc, bo = [clips[i] for i in rows], [owners[i] for i in rows]
        videos, frames, remapped, slab = batch_slabs(bc, bo)
        assert videos == sorted(set(bo)) and len(remapped) == len(slab) == len(bc)
        for k, v in enumerate(videos):
            used = {f for c, o in zip(bc, bo) if o == v for f in c.view.frames}
            assert frames[k] == sorted(used)                        # every decoded frame is read, each once
        for c, o, r, k in zip(bc, bo, remapped, slab):
            assert videos[k] == o
            assert [frames[k][i - 1] for i in r.view.frames] == c.view.frames
        for v, fr in zip(videos, frames):
            decoded.setdefault(v, []).extend(fr)
    for v, p in enumerate(plans):
        want = {f for c in p for f in c.view.frames}
        assert set(decoded[v]) == want
        if capacity >= 60:
            assert sorted(decoded[v]) == sorted(want)               # no video straddles: each frame decoded once
