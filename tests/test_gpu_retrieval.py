"""Nearest-neighbour video retrieval on the B200: the normalisation / similarity top-k / merge kernels bit-exact against
their float32 stand-ins (tests/emulate_retrieval.py) for every gallery split, cstp_b200.evaluate.video_features bit-exact
against per-video FinetuneEngine(n).forward_eval feature means, and the flow from a pretraining checkpoint to recall."""
import math
import os
import tempfile

import pytest
import torch

from tests.test_gpu_video_eval import FRAMES, LR, MOM, WD, _model, _synthetic_store
from tests.test_retrieval_cpu import _search, per_video_feature_means

pytestmark = pytest.mark.gpu


# ------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("k", [1, 50, 64])
def test_kernels_bit_exact_against_standins_for_every_split(k):
    from cstp_b200 import ops
    nq, ng, d = 300, 1237, 512                      # not multiples of the 64-query / 128-gallery tiles
    g = torch.Generator().manual_seed(k)
    q = torch.randn(nq, d, generator=g)
    gal = torch.randn(ng, d, generator=g)
    gal[900:1000] = gal[100:200]                    # duplicated rows: exact ties, resolved by the lower index
    q[10] = gal[150]                                # its two best neighbours tie at the top
    q[11] = 0                                       # a zero query: every similarity is 0
    gal[5] = 0
    ql = torch.randint(0, 20, (nq,), generator=g)
    gl = torch.randint(0, 20, (ng,), generator=g)
    cutoffs = [c for c in (1, 5, 10, 20, 50, 64) if c <= k]
    want_idx, want_sim, want_hits = _search(q, gal, k, 1, ql, gl, cutoffs)
    qd, gd = q.cuda(), gal.cuda()
    qn, gn = torch.empty_like(qd), torch.empty_like(gd)
    ops.l2_normalize_rows(qd, qn)
    ops.l2_normalize_rows(gd, gn)
    from tests import emulate_retrieval as E
    want_qn = torch.empty_like(q)
    E.l2_normalize_rows(q, want_qn)
    assert torch.equal(qn.cpu(), want_qn)
    host = ops.knn_splits(nq, ng)
    for splits in sorted({1, 7, host}):
        pv = torch.empty(splits, nq, k, device="cuda")
        pi = torch.empty(splits, nq, k, dtype=torch.int32, device="cuda")
        ops.knn_partial(qn, gn, k, splits, pv, pi)
        idx = torch.empty(nq, k, dtype=torch.int64, device="cuda")
        sim = torch.empty(nq, k, device="cuda")
        hits = torch.zeros(len(cutoffs), dtype=torch.int64, device="cuda")
        ops.knn_merge(pv, pi, idx, sim, ql.cuda(), gl.cuda(), torch.tensor(cutoffs, dtype=torch.int32, device="cuda"), hits)
        assert torch.equal(idx.cpu(), want_idx), splits
        assert torch.equal(sim.cpu(), want_sim), splits
        assert torch.equal(hits.cpu(), want_hits), splits
    assert not want_sim[11].any() and want_idx[11].tolist() == list(range(k))
    if k >= 2:
        assert want_idx[10, :2].tolist() == [150, 950] and want_sim[10, 0] == want_sim[10, 1]


def test_kernels_reject_out_of_range_arguments():
    from cstp_b200 import lib as L, ops
    q = torch.randn(4, 8, device="cuda")
    pv = torch.empty(1, 4, 65, device="cuda")
    pi = torch.empty(1, 4, 65, dtype=torch.int32, device="cuda")
    with pytest.raises(L.CstpError):
        ops.knn_partial(q, q, 65, 1, pv, pi)                        # k > 64
    with pytest.raises(L.CstpError):
        ops.knn_partial(q[:, :6].contiguous(), q[:, :6].contiguous(), 4, 1, pv[:, :, :4].contiguous(),
                        pi[:, :, :4].contiguous())                          # d % 4 != 0
    with pytest.raises(L.CstpError):
        ops.l2_normalize_rows(q.bfloat16(), torch.empty(4, 8, device="cuda"))       # the kernel reads fp32 rows


def test_retrieve_videos_rejects_mismatched_inputs_on_the_device():
    from cstp_b200.evaluate import retrieve_videos
    q, g = torch.randn(5, 8, device="cuda"), torch.randn(7, 8, device="cuda")
    for args in ((q, range(5), g, range(6)), (q, range(4), g, range(7)), (q.half(), range(5), g, range(7))):
        with pytest.raises(ValueError):
            retrieve_videos(*args, ks=(1, 5))
    r = retrieve_videos(q, torch.arange(5, device="cuda"), g, torch.arange(7, device="cuda"), ks=(1, 5))
    assert r["queries"] == 5 and r["neighbours"].shape == (5, 5)


# ------------------------------------------------------------------------------------------ video_features
def test_video_features_bit_exact_against_per_video_forward_eval():
    from oracle import cstp_oracle as O
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    from cstp_b200.data_process.gpu_clips import GpuClipPipeline
    from cstp_b200.evaluate import video_features
    n = len(FRAMES)
    store = _synthetic_store(n)
    m = _model().train()
    x = O.structured_batch(2, 0, 16, 112)[0].cuda()
    m.finetune_step(x, torch.tensor([3, 77], device="cuda"), lr=LR, momentum=MOM, weight_decay=WD)
    m.eval()
    runs = [video_features(m, store, FRAMES, capacity=3).cpu() for _ in range(2)]
    sampler, pipe = FinetuneClipSampler(16, 112, 4), GpuClipPipeline(16, 112)
    ref = per_video_feature_means(m, store, n, 16, 112, "cuda", lambda v: sampler.plan_test(FRAMES[v], 171, 128),
                                  pipe.assemble_clips)
    assert runs[0].shape == (n, 512)
    for v in range(n):
        assert torch.equal(runs[0][v], ref[v]), v
    assert torch.equal(runs[1], runs[0])


# ------------------------------------------------------------------------------------------ checkpoint -> recall
PALETTE = [(0, 0, 0), (255, 255, 255), (230, 20, 20), (20, 200, 30), (30, 40, 230), (240, 230, 20), (20, 220, 230),
           (220, 30, 220), (128, 128, 128), (250, 140, 0), (90, 40, 10), (10, 60, 90)]


def _videos(seeds, frames=48):
    """uint8 videos built to differ: per seed, its own colour from PALETTE under a moving grating of its own orientation
    and frequency."""
    t, y, x = torch.meshgrid(torch.arange(frames, dtype=torch.float32), torch.arange(128, dtype=torch.float32),
                             torch.arange(171, dtype=torch.float32), indexing="ij")
    out = []
    for s in seeds:
        a, f = 0.7 * s, 0.04 + 0.025 * (s % 7)
        wave = torch.sin(f * (x * math.cos(a) + y * math.sin(a)) + 0.3 * t)
        v = torch.tensor(PALETTE[s], dtype=torch.float32) + 25 * wave[..., None]
        out.append(v.clamp(0, 255).to(torch.uint8))
    return out


def _clips64(videos):
    """8-frame 64x64 pretraining clips (every other pixel) of the given videos, scaled to [-1, 1] like the clip pipeline."""
    return torch.stack([(v[:8, :128:2, 20:148:2].float() / 255 * 2 - 1).permute(3, 0, 1, 2) for v in videos])


def test_pretraining_checkpoint_to_retrieval_recall():
    from oracle import cstp_oracle as O
    from cstp_b200 import train
    from cstp_b200.data_process.datasets import GpuVideoStore
    from cstp_b200.evaluate import retrieve_videos, video_features
    from cstp_b200.models.model import neq_load_customized
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(0)
    pre = R21DBYOL(pretrain=True).cuda().train()
    # one training step, then lr-0 steps on the same clips until the BatchNorm running statistics have settled, as in
    # any real checkpoint: with the initial statistics (mean 0, variance 1) nothing is normalised in eval mode, the pooled
    # features are ~1e-10, and one step's shift of the running means (~1e-4) leaves every video the same feature
    labels = tuple(l.cuda() for l in O.structured_batch(2, 0, 8, 64)[2])
    x1, x2 = _clips64(_videos([0, 3])).cuda(), _clips64(_videos([1, 4])).cuda()
    pre.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=0.03)
    for _ in range(60):
        pre.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=0.0)
    path = os.path.join(tempfile.mkdtemp(), "epoch_1.pth.tar")
    train.save_checkpoint(path, pre, 0, "r21d_byol")
    sd = torch.load(path, map_location="cpu", weights_only=False)["state_dict"]
    sd = {k[len("module."):] if k.startswith("module.") else k: v for k, v in sd.items()}
    ft = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
    neq_load_customized(ft, sd, verbose=False)
    assert torch.equal(ft.state_dict()["online_net.conv1.spatial_conv.weight"], sd["online_net.conv1.spatial_conv.weight"])
    ft = ft.cuda().eval()

    n_gal, copies, unrelated = 10, [2, 5, 7], [10, 11]
    gallery, queries = GpuVideoStore(), GpuVideoStore()
    for v, vid in enumerate(_videos(range(n_gal))):
        gallery.put(v, vid.cuda())
    for i, vid in enumerate([gallery[c].cpu() for c in copies] + _videos(unrelated)):
        queries.put(i, vid.cuda())
    frames = 48
    g_feat = video_features(ft, gallery, [frames] * n_gal)
    q_feat = video_features(ft, queries, [frames] * len(copies + unrelated))
    g_labels = list(range(n_gal))
    q_labels = copies + [99] * len(unrelated)                        # unrelated videos have no class in the gallery
    r = retrieve_videos(q_feat, q_labels, g_feat, g_labels)
    assert r["queries"] == 5
    for i, c in enumerate(copies):
        assert torch.equal(q_feat[i], g_feat[c])
        assert r["neighbours"][i, 0] == c
        assert r["similarity"][i, 0] - r["similarity"][i, 1] > 1e-4         # the margin the top-1 check relies on
    assert r["recall"] == {k: 3 / 5 for k in (1, 5, 10, 20, 50)}
    assert (r["neighbours"][:, n_gal:] == -1).all() and torch.isneginf(r["similarity"][:, n_gal:]).all()
