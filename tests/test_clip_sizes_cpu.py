"""Clip geometries beyond 16 x 112 x 112 on the host side of the clip pipeline, without a GPU:
  * descriptors compiled at T in {32, 64} and S in {160, 224}, executed by the numpy stand-in of csrc/clip_pipeline.cu
    (tests/emulate_clips.py), equal the Pillow oracle byte for byte -- pretraining views (null and base chains: rotation,
    jitter, gray, blur, every 90-degree rotation label), finetune train / val / test views, frames of 171x128, 320x240
    and 340x256;
  * the launch layout `cstp_clip_assemble` picks (one CTA or a cluster pair per (frame, view)) and its capacity bound.
"""
import copy
import random
import re

import numpy as np
import pytest
import torch

from cstp_b200 import lib as L
from cstp_b200.data_process.clip_plan import FinetuneClipSampler, PretrainClipSampler
from cstp_b200.data_process.gpu_clips import clip_layout, compile_view
from oracle.clip_oracle import render_view, synthetic_video
from tests.emulate_clips import run_view
from tests.test_clip_pipeline import _force_base

FRAMES = [(171, 128), (320, 240), (340, 256)]
LIMIT = 226 * 1024


def seed_all(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


def pretrain_case(seed, T, S, w, h, variant="ucf", base=False):
    """A seeded pretraining plan at (T, S) on frames of w x h (base: both views get the full base chain), its video."""
    seed_all(seed)
    total = 2 * T + 7
    plan = PretrainClipSampler(T, S, variant).plan(total, w, h)
    if base:
        plan = _force_base(plan, seed)
    video = synthetic_video(total + 1, w, h, seed)
    return plan, video


def finetune_case(seed, T, S, mode, w, h, total=None):
    seed_all(seed)
    total = total or 3 * T
    s = FinetuneClipSampler(T, S, 4)
    plans = {"train": lambda: [s.plan_train(total, w, h)], "val": lambda: [s.plan_val(total, w, h)],
             "test": lambda: s.plan_test(total, w, h)}[mode]()
    return plans, synthetic_video(total + 1, w, h, seed)


def emulate(view, frame_base, video, S, n_frames=None):
    """The stand-in's clip for `view` (its first n_frames frames) and Pillow's, as (got, want)."""
    if n_frames is not None:
        view = copy.deepcopy(view)
        view.frames = view.frames[:n_frames]
        view.gray = view.gray[:n_frames] if view.gray is not None else None
    H, W = video.shape[1:3]
    d, coef, _ = compile_view(view, frame_base, W, H, S)
    got = torch.from_numpy(run_view(d, coef, video, len(view.frames), S))
    return got, render_view(view, video, frame_base, S)


@pytest.mark.parametrize("S", [160, 224])
@pytest.mark.parametrize("wh", FRAMES)
def test_pretraining_views_match_pillow(S, wh):
    w, h = wh
    for k, base in enumerate((False, True)):
        plan, video = pretrain_case(100 + S + w + k, 32, S, w, h, "ucf" if k == 0 else "kinetics", base)
        plan.views[0].rot, plan.views[1].rot = (2 * k) % 4, (2 * k + 1) % 4      # every rotation label over the pair
        for v in plan.views:                                                     # keep the box inside the rotated frame
            wr, hr = (h, w) if v.rot & 1 else (w, h)
            bw, bh = min(v.box[2] - v.box[0], wr), min(v.box[3] - v.box[1], hr)
            v.box = (wr - bw, hr - bh, wr, hr)
        for v in plan.views:
            got, want = emulate(v, plan.frame_base, video, S, n_frames=2)
            assert torch.equal(got, want), (S, wh, k, (got - want).abs().max().item())


def test_full_height_rotated_crop_at_224():
    """ROTATE_90 / ROTATE_270 of a 340x256 frame: a crop 340 rows tall, the tallest the samplers plan."""
    plan, video = pretrain_case(7, 16, 224, 340, 256, base=True)
    for v, rot in zip(plan.views, (1, 3)):
        v.rot, v.box = rot, (0, 0, 256, 340)
        got, want = emulate(v, plan.frame_base, video, 224, n_frames=1)
        assert torch.equal(got, want), rot
    assert clip_layout(224, 340)[0] == 2


def test_64_frame_clip_every_frame():
    """All 64 frames of a clip (frame numbers and per-frame gray channels fill the descriptor's arrays)."""
    plan, video = pretrain_case(3, 64, 160, 171, 128, base=True)
    v = plan.views[0]
    v.blur_sigma = None                                      # keeps the stand-in quick; blur is covered above
    v.gray = [(i * 7) % 3 for i in range(64)]
    d, coef, _ = compile_view(v, plan.frame_base, 171, 128, 160)
    assert list(d.frames) == [n - plan.frame_base for n in v.frames] and list(d.gray) == v.gray
    got, want = emulate(v, plan.frame_base, video, 160)
    assert got.shape == (3, 64, 160, 160) and torch.equal(got, want)
    with pytest.raises(ValueError):
        v.frames = v.frames + [v.frames[-1]]
        compile_view(v, plan.frame_base, 171, 128, 160)


@pytest.mark.parametrize("mode", ["train", "val", "test"])
@pytest.mark.parametrize("wh", FRAMES)
def test_finetune_views_match_pillow(mode, wh):
    w, h = wh
    for T in (32, 64):
        plans, video = finetune_case(40 + T + w, T, 224, mode, w, h, total=T * 5 if mode == "test" else None)
        if mode == "test":
            assert len(plans) > 1
        for p in plans[:2]:
            got, want = emulate(p.view, p.frame_base, video, 224, n_frames=2)
            assert torch.equal(got, want), (mode, wh, T)


def test_finetune_train_views_at_160_and_jitter():
    for seed in range(6):                                   # ClipColorJitter fires with p = 0.3: some of these carry it
        plans, video = finetune_case(seed, 32, 160, "train", 320, 240)
        got, want = emulate(plans[0].view, plans[0].frame_base, video, 160, n_frames=2)
        assert torch.equal(got, want), seed
    seed_all(0)
    with pytest.raises(ValueError):                          # img_val / img_test exist for 112 and 224 only
        FinetuneClipSampler(16, 160).plan_val(40, 320, 240)


def _align(n):
    return (n + 15) & ~15


def expected_layout(S, h):
    row = S * 3
    one = _align(h * row) + 2 * _align(S * row)
    if one <= LIMIT:
        return 1, one
    hs = (S + 1) // 2
    pair = _align(max((h + 1) // 2, hs) * row) + _align(hs * row)
    return (2, pair) if pair <= LIMIT else (None, pair)


def test_layout_matches_the_capacity_formulas():
    for S in (8, 57, 112, 129, 160, 180, 223, 224):
        for h in list(range(1, 1400, 37)) + [S, 2 * S, 340, 464, 465]:
            want = expected_layout(S, h)
            if want[0] is None:
                with pytest.raises(L.CstpError):
                    clip_layout(S, h)
            else:
                assert clip_layout(S, h) == want, (S, h)


@pytest.mark.parametrize("S, one_max, pair_max", [(112, 464, 1264), (160, 162, 804), (224, 0, 464)])
def test_layout_edges(S, one_max, pair_max):
    """The tallest crop each variant holds, and one row more."""
    if one_max:
        assert clip_layout(S, one_max)[0] == 1
    assert clip_layout(S, one_max + 1)[0] == 2
    assert clip_layout(S, pair_max)[0] == 2 and clip_layout(S, pair_max)[1] <= LIMIT
    with pytest.raises(L.CstpError) as e:
        clip_layout(S, pair_max + 1)
    msg = str(e.value)
    m = re.search(r"invalid argument: crop height (\d+) needs (\d+) bytes of shared memory \(limit (\d+)\)", msg)
    assert m and int(m.group(1)) == pair_max + 1 and int(m.group(2)) > LIMIT and int(m.group(3)) == LIMIT, msg


def test_layout_rejects_sizes_outside_the_kernel():
    for S in (7, 225):
        with pytest.raises(L.CstpError):
            clip_layout(S, 100)
    assert L.CSTP_CLIP_T == 64 and L.CSTP_CLIP_S == 224
