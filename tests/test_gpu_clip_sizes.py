"""Clip geometries beyond 16 x 112 x 112 on the B200:
  * csrc/clip_pipeline.cu against the Pillow oracle, bit for bit: every view kind at S = 224 (the cluster-pair kernel),
    64-frame clips, and S = 160 with one batch on each side of the one-CTA / pair choice;
  * the finetune engine per layer at (B, T, S) = (2, 16, 224) and (2, 32, 112), its loss against the fp32 oracle, and
    one pretraining step at 16 x 224 against the fp32 oracle;
  * an inference engine of capacity 60 at 16 x 224 (tensors past 2^31 bytes) against the same clips 4 at a time;
  * the batch sources and video-level evaluation at sample_size 224.
"""
import os

import numpy as np
import pytest
import torch

from cstp_b200.data_process.gpu_clips import GpuClipPipeline, clip_layout
from oracle.clip_oracle import render_view
from tests.test_clip_sizes_cpu import FRAMES, finetune_case, pretrain_case, seed_all

pytestmark = pytest.mark.gpu
LR, MOM, WD = 0.025, 0.9, 1e-3


def _pretrain_batch(T, S, seed, n=6):
    """n pretraining plans over the three frame sizes, alternately with the full base chain, every rotation label, and
    for the 340x256 frames ROTATE_90 / ROTATE_270 crops of the full 340-row height."""
    plans, vids = [], []
    for b in range(n):
        w, h = FRAMES[b % 3]
        plan, video = pretrain_case(seed + b, T, S, w, h, "ucf" if b % 2 == 0 else "kinetics", base=b % 2 == 1)
        plan.views[0].rot, plan.views[1].rot = b % 4, (b + 1) % 4
        for v in plan.views:
            wr, hr = (h, w) if v.rot & 1 else (w, h)
            bw, bh = min(v.box[2] - v.box[0], wr), min(v.box[3] - v.box[1], hr)
            v.box = (wr - bw, hr - bh, wr, hr)
            if (w, h) == (340, 256) and v.rot & 1:
                v.box = (0, 0, 256, 340)
        plans.append(plan)
        vids.append(video)
    return plans, vids


def _check_pretrain(plans, vids, T, S):
    pipe = GpuClipPipeline(T, S)
    x1, x2 = pipe.assemble(plans, [torch.from_numpy(v).cuda() for v in vids])
    torch.cuda.synchronize()
    for b, (plan, vid) in enumerate(zip(plans, vids)):
        for k, x in enumerate((x1, x2)):
            want = render_view(plan.views[k], vid, plan.frame_base, S)
            got = x[b].cpu()
            assert torch.equal(got, want), (T, S, b, k, (got - want).abs().max().item(), (got != want).sum().item())
    return max(v.box[3] - v.box[1] if v.resize is None else vid.shape[1] for p, vid in zip(plans, vids) for v in p.views)


def test_pretraining_views_at_224_bit_exact():
    plans, vids = _pretrain_batch(16, 224, 500)
    assert _check_pretrain(plans, vids, 16, 224) == 340 and clip_layout(224, 340)[0] == 2


def test_64_frame_clips_bit_exact():
    plans, vids = _pretrain_batch(64, 224, 600, n=2)
    _check_pretrain(plans, vids, 64, 224)
    plans, vids = _pretrain_batch(64, 112, 700, n=2)
    _check_pretrain(plans, vids, 64, 112)


def test_both_variants_at_160():
    """S = 160: a batch whose crops fit one CTA (<= 162 rows) and one that needs the pair, both equal to Pillow."""
    small, vids_s = _pretrain_batch(16, 160, 800, n=3)
    for p in small:
        for v in p.views:
            if v.box[3] - v.box[1] > 150:
                v.box = (v.box[0], v.box[3] - 150, v.box[2], v.box[3])
    big, vids_b = _pretrain_batch(16, 160, 900, n=3)
    for plans, vids, cluster in ((small, vids_s, 1), (big, vids_b, 2)):
        h = _check_pretrain(plans, vids, 16, 160)
        assert clip_layout(160, h)[0] == cluster, h


@pytest.mark.parametrize("mode", ["train", "val", "test"])
def test_finetune_views_at_224_bit_exact(mode):
    pipe = GpuClipPipeline(16, 224)
    for k, (w, h) in enumerate(FRAMES):
        plans, video = finetune_case(900 + k, 16, 224, mode, w, h)
        plans = plans[:4]
        out = pipe.assemble_clips(plans, [torch.from_numpy(video).cuda()] * len(plans))
        torch.cuda.synchronize()
        for j, p in enumerate(plans):
            assert torch.equal(out[j].cpu(), render_view(p.view, video, p.frame_base, 224)), (mode, w, h, j)


# ------------------------------------------------------------------------------------------ engines
def _ft_model(record=False):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
    m.engine_options = {"record": record}
    return m


@pytest.mark.parametrize("B,T,S", [(2, 16, 224), (2, 32, 112)])
def test_finetune_engine_per_layer_and_oracle(B, T, S):
    from oracle import cstp_oracle as O
    from tests import local_parity as LP
    x = O.structured_batch(B, 0, T, S)[0]
    labels = torch.tensor([3, 77])
    m = _ft_model(record=True)
    before = {k: v.clone() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    trainable = [n for n, _ in m.named_parameters()]
    m.cuda().train()
    opt = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    logits = m(x.cuda(), o_type="ft_all")
    loss = torch.nn.CrossEntropyLoss()(logits, labels.cuda())
    opt.zero_grad()
    loss.backward()
    res = LP.check_conv_units(m._engine, before, "online")
    w = LP.worst(res)
    print(f"worst per-layer error at {B}x{T}x{S}:", w)
    assert len([t for t in res if t.startswith("online.")]) == 24 and w[0] < 1e-2, w
    torch.set_num_threads(os.cpu_count() or 1)
    r = O.finetune_step({k: v.clone() for k, v in before.items()}, trainable, x, labels, LR, {}, MOM, WD)
    assert abs(loss.item() - r["loss"]) < 3e-3 * r["loss"], (loss.item(), r["loss"])


def test_pretraining_step_at_224_against_oracle():
    from oracle import cstp_oracle as O
    from cstp_b200.engine import trainable_param_specs
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    model = R21DBYOL(pretrain=True)
    state = {k: v.clone() for k, v in model.state_dict().items() if not k.endswith("num_batches_tracked")}
    x1, x2, labels = O.structured_batch(2, 0, 16, 224)
    model.cuda()
    got = model.train_step(x1.cuda(), x2.cuda(), tuple(l.cuda() for l in labels), (0.1, 1, 1, 1, 1), lr=0.03).cpu()
    torch.set_num_threads(os.cpu_count() or 1)
    ref = O.pretrain_step(state, [n for n, _ in trainable_param_specs()], x1, x2, labels, [0.1, 1, 1, 1, 1], 0.03, {})
    total = 0.1 * got[7].item() + got[6].item()
    assert abs(total - ref["loss_total"]) < 1e-3 * abs(ref["loss_total"]), (total, ref["loss_total"])


def _trained_ft_model(T=16, S=112):
    from oracle import cstp_oracle as O
    m = _ft_model().cuda().train()
    x = O.structured_batch(2, 0, T, S)[0].cuda()
    m.finetune_step(x, torch.tensor([3, 77], device="cuda"), lr=LR, momentum=MOM, weight_decay=WD)
    return m.eval()


def test_inference_engine_past_2_31_bytes_equals_small_batches():
    """Capacity 60 at 16 x 224: its largest activations exceed 2^31 bytes.  Eval rows are independent, so any 32-bit
    offset that wraps shows up as a mismatch against the same clips run 4 at a time."""
    m = _trained_ft_model()
    x = (torch.rand(60, 3, 16, 224, 224, generator=torch.Generator().manual_seed(3)) * 2 - 1).cuda()
    assert 60 * 16 * 112 * 112 * 144 * 2 > 2 ** 31          # one conv2 tensor of 144 bf16 channels on 112 x 112 planes
    with torch.no_grad():
        big = m.inference_engine(60, 16, 224, 224, "cuda")
        m._repack_if_changed(big)
        got = big.forward_batch(x)[:60, :101].clone()
        small = m.inference_engine(4, 16, 224, 224, "cuda")
        m._repack_if_changed(small)
        want = torch.cat([small.forward_batch(x[i:i + 4])[:4, :101].clone() for i in range(0, 60, 4)])
    assert torch.isfinite(got).all() and torch.equal(got, want), (got - want).abs().max().item()


# ------------------------------------------------------------------------------------------ batch sources, evaluation
def test_jpeg_finetune_batches_at_224_equal_store_batches():
    from cstp_b200.data_process.datasets import FinetuneBatches, JpegFinetuneBatches
    from tests.test_gpu_finetune_batches import COUNTS, LABELS, SIZES, _collect, _dataset
    store, read_frames, _ = _dataset(COUNTS, SIZES)
    for split in ("train", "val"):
        kw = dict(batch_size=3, split=split, seed=4, sample_size=224)
        ref = FinetuneBatches(store, COUNTS, LABELS, **kw)
        src = JpegFinetuneBatches(read_frames, COUNTS, LABELS, **kw)
        for epoch in range(2):
            seed_all(20 + epoch)
            want = _collect(ref, epoch)
            seed_all(20 + epoch)
            got = _collect(src, epoch)
            assert len(got) == len(want) > 0 and got[0][0].shape[-3:] == (16, 224, 224)
            for (a, la), (b, lb) in zip(got, want):
                assert torch.equal(a, b) and torch.equal(la, lb)


def test_evaluation_at_224_equals_per_video_forward_eval():
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    from cstp_b200.evaluate import test_videos, test_videos_jpeg, video_features, video_features_jpeg
    from tests.test_gpu_finetune_batches import EVAL_FRAMES, EVAL_SIZES, _dataset
    from tests.test_retrieval_cpu import per_video_feature_means
    from tests.test_gpu_video_eval import _reference_logits, seq_sum
    frames, sizes = EVAL_FRAMES[:5], EVAL_SIZES[:5]                  # 29 and 130 frames: one window up to eight
    store, read_frames, _ = _dataset(frames, sizes)
    m = _trained_ft_model()
    n = len(frames)
    labels = [int(v) for v in torch.randint(0, 101, (n,), generator=torch.Generator().manual_seed(4))]
    sampler, pipe = FinetuneClipSampler(16, 224, 4), GpuClipPipeline(16, 224)
    means = []
    with torch.no_grad():
        for v in range(n):
            plans = sampler.plan_test(frames[v], *sizes[v])
            clips = pipe.assemble_clips(plans, [store[v]] * len(plans))
            means.append(seq_sum(_reference_logits(m, clips, 16, 224).cpu()) / float(len(plans)))
    got = test_videos(m, store, frames, labels, sample_size=224, capacity=5, keep_logits=True)
    assert torch.equal(got["logits"], torch.stack(means))
    jp = test_videos_jpeg(m, read_frames, frames, labels, sample_size=224, capacity=5, keep_logits=True)
    assert torch.equal(jp["logits"], got["logits"]) and torch.equal(jp["predictions"], got["predictions"])
    assert (jp["hits"], jp["clips"]) == (got["hits"], got["clips"])
    feats = video_features(m, store, frames, sample_size=224, capacity=5).cpu()
    ref = per_video_feature_means(m, store, n, 16, 224, "cuda", lambda v: sampler.plan_test(frames[v], *sizes[v]),
                                  pipe.assemble_clips)
    for v in range(n):
        assert torch.equal(feats[v], ref[v]), v
    assert torch.equal(video_features_jpeg(m, read_frames, frames, sample_size=224, capacity=5, sizes=sizes).cpu(), feats)


def test_finetune_epochs_and_test_videos_jpeg_at_224():
    """INTEGRATION.md's 224 path end to end: JpegFinetuneBatches(sample_size=224) -> finetune_epochs ->
    test_videos_jpeg(sample_size=224), whose results equal the store-fed test_videos at 224."""
    import tempfile
    import types
    from cstp_b200 import train
    from cstp_b200.data_process.datasets import JpegFinetuneBatches
    from cstp_b200.evaluate import test_videos, test_videos_jpeg
    from tests.test_gpu_finetune_batches import COUNTS, LABELS, SIZES, _dataset
    store, read_frames, _ = _dataset(COUNTS, SIZES)
    tr = JpegFinetuneBatches(read_frames, COUNTS, LABELS, 2, split="train", sample_size=224, seed=1)
    va = JpegFinetuneBatches(read_frames, COUNTS, LABELS, 2, split="val", sample_size=224)
    opts = types.SimpleNamespace(n_epochs=1, learning_rate=LR, momentum=MOM, weight_decay=WD, lr_patience=0,
                                 task="ft_all", highest_val={"name": -1.0})
    seed_all(11)
    m = _ft_model().cuda()
    rows_t, rows_v = train.finetune_epochs(m, tr, va, opts, result_path=tempfile.mkdtemp())
    assert len(rows_t) == len(rows_v) == 1 and np.isfinite(rows_t[0]["loss"]) and np.isfinite(rows_v[0]["loss"])
    m.eval()
    got = test_videos_jpeg(m, read_frames, COUNTS, LABELS, sample_size=224, capacity=8, keep_logits=True)
    want = test_videos(m, store, COUNTS, LABELS, sample_size=224, capacity=8, keep_logits=True)
    assert got["videos"] == len(COUNTS) and torch.isfinite(got["logits"]).all()
    assert torch.equal(got["logits"], want["logits"]) and got["hits"] == want["hits"]
