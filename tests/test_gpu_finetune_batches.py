"""Finetune / validation batch sources and JPEG-fed evaluation on the B200: `FinetuneBatches` against `assemble_clips` on
the same plans, `JpegFinetuneBatches` against `FinetuneBatches` over Pillow-decoded copies of the same JPEG frames, the
decode-error contract, `test_videos_jpeg` / `video_features_jpeg` against the store-fed calls, and a pretraining
checkpoint finetuned for two epochs from JPEG frames with the same log rows as from a store."""
import os
import random
import tempfile
import types

import numpy as np
import pytest
import torch
from PIL import features

from cstp_b200.data_process.clip_plan import FinetuneClipSampler
from cstp_b200.data_process.datasets import (FinetuneBatches, GpuVideoStore, JpegFinetuneBatches,
                                             distributed_indices)
from cstp_b200.data_process.gpu_clips import GpuClipPipeline
from tests import jpeg_cases as J

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not features.check_feature("libjpeg_turbo"),
                                                  reason="the decode contract is Pillow on libjpeg-turbo")]
LR, MOM, WD = 0.025, 0.9, 1e-3


def _dataset(counts, sizes):
    """JPEG videos of the given lengths and frame sizes (frames numbered from 1), a store of their Pillow decodes, and
    a read_frames that records every read."""
    enc = []
    store = GpuVideoStore("cuda")
    for i, ((w, h), n) in enumerate(zip(sizes, counts)):
        frames = J.content("video", w, h, i)
        video = [np.roll(np.roll(frames, 5 * k, axis=1), 2 * k, axis=0) for k in range(n)]
        enc.append([J.pil_encode(f, ("420", "422", "444")[i % 3], quality=85 + i % 10) for f in video])
        store.put(i, np.stack([J.pillow_decode(b) for b in enc[i]]))
    reads = []

    def read_frames(video, frame_numbers):
        reads.append((video, list(frame_numbers)))
        return [enc[video][f - 1] for f in frame_numbers]
    return store, read_frames, reads


SIZES = [(171, 128), (160, 121), (173, 131), (171, 128), (149, 113), (171, 128), (161, 120)]
COUNTS = [48, 61, 37, 70, 44, 20, 66]                  # 37, 44 and 20 frames: the clip wraps around
LABELS = [5, 17, 99, 0, 42, 64, 100]


def _seed(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


def _collect(src, epoch):
    return [(x.clone(), y.clone()) for x, y in src(epoch)]


@pytest.mark.parametrize("split", ["train", "val"])
def test_finetune_batches_equal_assemble_clips_on_the_same_plans(split):
    store, _, _ = _dataset(COUNTS, SIZES)
    src = FinetuneBatches(store, COUNTS, LABELS, 3, split=split, seed=2)
    sampler, pipe = FinetuneClipSampler(16, 112, 4), GpuClipPipeline(16, 112)
    draw = sampler.plan_train if split == "train" else sampler.plan_val
    for epoch in range(2):
        _seed(epoch)
        got = _collect(src, epoch)
        _seed(epoch)
        order = distributed_indices(len(COUNTS), epoch, 0, 1, 2, split == "train")
        ids = [order[k:k + 3] for k in range(0, len(order), 3)]
        ids = [b for b in ids if len(b) == 3] if split == "train" else ids
        assert len(got) == len(ids) == (2 if split == "train" else 3)
        for (x, y), b in zip(got, ids):
            plans = [draw(COUNTS[i], SIZES[i][0], SIZES[i][1]) for i in b]
            assert torch.equal(x, pipe.assemble_clips(plans, [store[i] for i in b]))
            assert y.dtype == torch.int64 and y.device.type == "cuda" and y.tolist() == [LABELS[i] for i in b]


@pytest.mark.parametrize("split", ["train", "val"])
@pytest.mark.parametrize("rank,world", [(0, 1), (1, 2)])
def test_jpeg_finetune_batches_equal_store_batches(split, rank, world):
    store, read_frames, reads = _dataset(COUNTS, SIZES)
    kw = dict(batch_size=2, split=split, rank=rank, world=world, seed=3)
    ref = FinetuneBatches(store, COUNTS, LABELS, **kw)
    src = JpegFinetuneBatches(read_frames, COUNTS, LABELS, **kw)
    n = 0
    for epoch in range(2):
        _seed(10 + epoch)
        want = _collect(ref, epoch)
        _seed(10 + epoch)
        got = _collect(src, epoch)
        assert len(got) == len(want) > 0
        for (a, la), (b, lb) in zip(got, want):
            assert torch.equal(a, b) and torch.equal(la, lb)
            n += 1
    assert n >= 4
    assert all(fr == sorted(set(fr)) for _, fr in reads)          # no frame read twice for one clip


def test_jpeg_finetune_batches_raise_at_the_next_request():
    _, read_frames, _ = _dataset(COUNTS[:4], SIZES[:4])

    def broken(video, frame_numbers):
        out = read_frames(video, frame_numbers)
        return [b[:60] if video == 2 else b for b in out]
    src = JpegFinetuneBatches(broken, COUNTS[:4], LABELS[:4], 1, split="val", sizes=SIZES[:4])
    it = src(0)
    next(it), next(it), next(it)                       # videos 0, 1, 2: the third batch holds the bad frames
    with pytest.raises(ValueError, match=r"video 2 frame \d+: malformed"):
        next(it)


# ------------------------------------------------------------------------------------------ evaluation
EVAL_FRAMES = [29, 95, 200, 61, 130, 45, 64, 250]       # 29 and 45: shorter than one test window
EVAL_SIZES = [(171, 128), (160, 121), (171, 128), (173, 131), (171, 128), (149, 113), (171, 128), (171, 128)]


def _finetuned_model():
    from oracle import cstp_oracle as O
    from tests.test_gpu_video_eval import _model
    m = _model().train()
    x = O.structured_batch(2, 0, 16, 112)[0].cuda()
    m.finetune_step(x, torch.tensor([3, 77], device="cuda"), lr=LR, momentum=MOM, weight_decay=WD)
    return m.eval()


def test_jpeg_fed_evaluation_equals_store_fed():
    from cstp_b200.evaluate import test_videos, test_videos_jpeg, video_features, video_features_jpeg
    store, read_frames, reads = _dataset(EVAL_FRAMES, EVAL_SIZES)
    m = _finetuned_model()
    n = len(EVAL_FRAMES)
    labels = [int(v) for v in torch.randint(0, 101, (n,), generator=torch.Generator().manual_seed(4))]
    sampler = FinetuneClipSampler(16, 112, 4)
    used = [{f for c in sampler.plan_test(t, w, h) for f in c.view.frames} for t, (w, h) in zip(EVAL_FRAMES, EVAL_SIZES)]
    for capacity in (3, 7, 60):
        want = test_videos(m, store, EVAL_FRAMES, labels, capacity=capacity, keep_logits=True)
        reads.clear()
        got = test_videos_jpeg(m, read_frames, EVAL_FRAMES, labels, capacity=capacity, keep_logits=True)
        assert torch.equal(got["logits"], want["logits"]), capacity
        assert torch.equal(got["predictions"], want["predictions"]), capacity
        assert (got["hits"], got["videos"], got["clips"]) == (want["hits"], want["videos"], want["clips"])
        assert reads[:n] == [(v, [1]) for v in range(n)]          # planning reads each video's first frame once
        for v in range(n):
            got_frames = [f for video, fr in reads[n:] if video == v for f in fr]
            assert set(got_frames) == used[v]                      # every frame a window reads, and no other
            if capacity == 60:
                assert len(got_frames) == len(used[v])             # one batch: each frame decoded once
        assert torch.equal(video_features_jpeg(m, read_frames, EVAL_FRAMES, capacity=capacity, sizes=EVAL_SIZES),
                           video_features(m, store, EVAL_FRAMES, capacity=capacity)), capacity
    assert want["clips"] > 2 * 7


def test_jpeg_fed_evaluation_names_a_rejected_frame():
    from cstp_b200.evaluate import test_videos_jpeg
    _, read_frames, _ = _dataset(EVAL_FRAMES[:3], EVAL_SIZES[:3])

    def broken(video, frame_numbers):
        return [b[:60] if (video, f) == (1, 61) else b for f, b in zip(frame_numbers, read_frames(video, frame_numbers))]
    with pytest.raises(ValueError, match=r"video 1 frame 61: malformed"):
        test_videos_jpeg(_finetuned_model(), broken, EVAL_FRAMES[:3], [0, 1, 2], capacity=60, sizes=EVAL_SIZES[:3])


# ------------------------------------------------------------------------------------------ checkpoint -> finetune
def test_pretraining_checkpoint_finetunes_from_jpeg_frames_like_from_a_store():
    from oracle import cstp_oracle as O
    from cstp_b200 import train
    from cstp_b200.models.model import neq_load_customized
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from tests.test_gpu_retrieval import _clips64, _videos
    torch.manual_seed(0)
    pre = R21DBYOL(pretrain=True).cuda().train()
    labels = tuple(l.cuda() for l in O.structured_batch(2, 0, 8, 64)[2])
    x1, x2 = _clips64(_videos([0, 3])).cuda(), _clips64(_videos([1, 4])).cuda()
    for lr in (0.03, 0.0, 0.0):
        pre.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=lr)
    d = tempfile.mkdtemp()
    ckpt = os.path.join(d, "save_1.pth")
    train.save_checkpoint(ckpt, pre, 0, "r21d_byol")

    def finetune_model():
        sd = torch.load(ckpt, map_location="cpu", weights_only=False)["state_dict"]
        sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}
        torch.manual_seed(5)                            # the head is initialised, not loaded
        ft = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
        neq_load_customized(ft, sd, verbose=False)
        return ft.cuda()

    n_train, n_val = 9, 5
    counts, sizes = COUNTS + [52, 80, 33, 47, 90, 29, 58], SIZES * 2
    store, read_frames, _ = _dataset(counts[:n_train + n_val], sizes[:n_train + n_val])
    lab = [(7 * i) % 101 for i in range(n_train + n_val)]
    val_ids = list(range(n_train, n_train + n_val))

    def val_read(video, frame_numbers):
        return read_frames(val_ids[video], frame_numbers)
    val_store = GpuVideoStore("cuda")
    for k, v in enumerate(val_ids):
        val_store.put(k, store[v])
    runs = {}
    for name in ("store", "jpeg"):
        if name == "store":
            tr = FinetuneBatches(store, counts[:n_train], lab[:n_train], 4, split="train", seed=1)
            va = FinetuneBatches(val_store, counts[n_train:n_train + n_val], lab[n_train:], 4, split="val")
        else:
            tr = JpegFinetuneBatches(read_frames, counts[:n_train], lab[:n_train], 4, split="train", seed=1)
            va = JpegFinetuneBatches(val_read, counts[n_train:n_train + n_val], lab[n_train:], 4, split="val")
        out = os.path.join(d, name)
        os.mkdir(out)
        opts = types.SimpleNamespace(n_epochs=2, learning_rate=LR, momentum=MOM, weight_decay=WD, lr_patience=0,
                                     task="ft_all", highest_val={"name": -1.0})
        _seed(11)
        rows = train.finetune_epochs(finetune_model(), tr, va, opts, result_path=out)
        runs[name] = (rows, sorted(os.listdir(out)), opts.highest_val)
    (rows_t, rows_v), files, best = runs["jpeg"]
    assert runs["jpeg"][0] == runs["store"][0]                     # identical train and val rows, bit for bit
    assert [r["epoch"] for r in rows_t] == [1, 2] == [r["epoch"] for r in rows_v]
    assert all(np.isfinite(r["loss"]) for r in rows_t + rows_v)
    assert files == runs["store"][1] == [next(iter(best))] and files[0] in ("save_1_max.pth", "save_2_max.pth")
    ck = torch.load(os.path.join(d, "jpeg", files[0]), weights_only=False)
    assert set(ck) == {"epoch", "arch", "state_dict", "optimizer"}
