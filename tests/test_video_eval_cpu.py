"""Video-level test evaluation on CPU: the CPU stand-ins of cstp_video_accumulate / cstp_video_finalize against torch,
cstp_b200.evaluate.test_videos (clips of consecutive videos packed into full batches of one inference engine) against the
drop-in per-video loop of test.py:76-93, and the drop-in's inference engines (engines built, training state untouched,
re-packing after optimizer.step), all over the CPU emulator (tests/emulate_ops.py, tests/emulate_video_eval.py) in fp32."""
import os
import re
import tempfile
from pathlib import Path

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import cstp_oracle as O

ROOT = Path(__file__).resolve().parents[1]
T_CLIP = 4
LR, MOM, WD = 0.025, 0.9, 1e-3


@pytest.fixture()
def emu():
    from cstp_b200 import engine
    from tests import emulate_video_eval
    saved = engine.ops, engine.ACT_DTYPE
    engine.ops, engine.ACT_DTYPE = emulate_video_eval, torch.float32
    try:
        yield engine
    finally:
        engine.ops, engine.ACT_DTYPE = saved


def _model(seed=1):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(seed)
    return R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)


def seq_mean(rows):
    """Mean over clips the way the kernels define it: a sequential fp32 sum in clip order, divided by the count."""
    acc = rows[0].clone()
    for r in rows[1:]:
        acc += r
    return acc / float(rows.shape[0])


def ranked(mean, k):
    """Class indices by value, descending, ties to the lower index."""
    return [c for _, c in sorted((-v, c) for c, v in enumerate(mean.tolist()))][:k]


# ------------------------------------------------------------------------------------------ stand-in semantics
def _score(logits, counts, capacity, labels, k=5):
    """Feeds logits [clips][ld] batch by batch through the stand-ins with evaluate.batch_tables' work lists."""
    from cstp_b200.evaluate import batch_tables
    from tests import emulate_video_eval as E
    n_cls = 101
    tab = torch.from_numpy(batch_tables(counts, capacity))
    sums = torch.zeros(len(counts), n_cls)
    mean = torch.zeros(len(counts), n_cls)
    topk = torch.zeros(len(counts), k, dtype=torch.int64)
    hits = torch.zeros(2, dtype=torch.int64)
    for b in range(tab.shape[0]):
        rows = logits[b * capacity:(b + 1) * capacity]
        buf = torch.full((capacity, logits.shape[1]), float("nan"))          # padding rows must never be read
        buf[:rows.shape[0]] = rows
        E.video_accumulate(buf, n_cls, tab[b, 0], sums, rows=rows.shape[0])
        E.video_finalize(sums, tab[b, 1], topk, torch.tensor(labels), mean, hits)
    assert not sums.any()                                                   # finalized slots are left zero
    return mean, topk, hits


@pytest.mark.parametrize("capacity", [1, 3, 7, 60])
def test_standins_match_torch_mean_and_topk(capacity):
    g = torch.Generator().manual_seed(5)
    counts = [1, 4, 1, 9, 2, 13, 1]                 # single-clip videos and videos straddling batch boundaries
    logits = torch.randn(sum(counts), 112, generator=g)
    labels = [int(v) for v in torch.randint(0, 101, (len(counts),), generator=g)]
    mean, topk, hits = _score(logits, counts, capacity, labels)
    h1 = h5 = 0
    start = 0
    for v, n in enumerate(counts):
        rows = logits[start:start + n, :101]
        start += n
        ref = seq_mean(rows)
        assert torch.equal(mean[v], ref)
        assert torch.allclose(mean[v], rows.mean(0), rtol=1e-6, atol=1e-6)
        assert topk[v].tolist() == torch.topk(ref, 5).indices.tolist()    # no ties in random data
        h1 += int(topk[v, 0] == labels[v])
        h5 += int(labels[v] in topk[v].tolist())
    assert hits.tolist() == [h1, h5]


def test_standin_ties_go_to_the_lower_class_index():
    logits = torch.zeros(2, 112)
    logits[:, [7, 3, 50, 9]] = 2.0                  # four-way tie at the top, then a tie between 20 and 11
    logits[:, [20, 11]] = 1.0
    mean, topk, hits = _score(logits, [2], 60, [9], k=8)
    assert topk[0].tolist() == [3, 7, 9, 50, 11, 20, 0, 1]
    assert hits.tolist() == [0, 1]


# ------------------------------------------------------------------------------------------ test_videos
FRAMES = [29, 13, 5, 61, 40, 17, 90, 29]


def _store(n):
    from cstp_b200.data_process.datasets import GpuVideoStore
    store = GpuVideoStore(device="cpu")
    for v in range(n):
        f = torch.zeros(FRAMES[v], 8, 12, 3, dtype=torch.uint8)
        f[0, 0, 0, 0] = v                           # the fake assembler's video tag
        store.put(v, f)
    return store


def fake_assemble(plans, videos, out):
    """Seeded clips that depend only on (video, frame window): the same clip whichever batch it lands in."""
    for i, (p, vid) in enumerate(zip(plans, videos)):
        g = torch.Generator().manual_seed(1000 * int(vid[0, 0, 0, 0]) + p.view.frames[0])
        out[i] = torch.rand(out.shape[1:], generator=g) * 2 - 1
    return out


def per_video_loop(m, store, n, labels):
    """The drop-in loop of test.py:76-93: one video per batch, mean over its clips, top-5."""
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    sampler = FinetuneClipSampler(T_CLIP, 112, 4)
    means, preds, hits = [], [], [0, 0]
    with torch.no_grad():
        for v in range(n):
            plans = sampler.plan_test(FRAMES[v], 12, 8)
            clips = fake_assemble(plans, [store[v]] * len(plans), torch.empty(len(plans), 3, T_CLIP, 112, 112))
            mean = seq_mean(m(clips, None, o_type="test"))
            top = ranked(mean, 5)
            means.append(mean)
            preds.append(top)
            hits[0] += int(top[0] == labels[v])
            hits[1] += int(labels[v] in top)
    return torch.stack(means), torch.tensor(preds), hits


def test_test_videos_packing_equals_per_video_loop(emu):
    from cstp_b200.evaluate import test_videos
    n = len(FRAMES)
    store = _store(n)
    m = _model()
    m.eval()
    ref_mean, ref_pred, ref_hits = per_video_loop(m, store, n, list(range(n)))
    labels = [int(p[0]) if v % 2 else int(p[3]) for v, p in enumerate(ref_pred)]   # top-1 / top-5 hits and misses
    labels[0] = 100 if 100 not in ref_pred[0].tolist() else 99
    ref_hits = [sum(int(ref_pred[v, 0] == labels[v]) for v in range(n)),
                sum(int(labels[v] in ref_pred[v].tolist()) for v in range(n))]
    r = test_videos(m, store, FRAMES[:n], labels, sample_duration=T_CLIP, capacity=7, keep_logits=True,
                    assemble=fake_assemble)
    # the CPU stand-in's fp32 GEMMs block differently for different batch sizes, so a clip's logits here depend on its
    # batch in the last bits (the sm_100a kernels do not: tests/test_gpu_video_eval.py compares bits)
    assert torch.allclose(r["logits"], ref_mean, rtol=1e-5, atol=1e-6)
    assert torch.equal(r["predictions"], ref_pred)
    assert r["hits"] == tuple(ref_hits) and 0 < ref_hits[0] < ref_hits[1] < n
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    clips = sum(len(FinetuneClipSampler(T_CLIP, 112, 4).plan_test(f, 12, 8)) for f in FRAMES[:n])
    assert r["videos"] == n and r["clips"] == clips and clips > 2 * 7          # several batches, videos straddling them
    assert r["top1"] == ref_hits[0] / n and r["top5"] == ref_hits[1] / n


# ------------------------------------------------------------------------------------------ engines of the drop-in
def _count_builds(monkeypatch):
    from cstp_b200 import engine
    built = []
    init = engine.ProgramEngine.__init__

    def spy(self, B, *a, **k):
        built.append((type(self).__name__, B))
        init(self, B, *a, **k)
    monkeypatch.setattr(engine.ProgramEngine, "__init__", spy)
    return built


def test_eval_batches_build_only_bucket_engines_and_leave_training_alone(emu, monkeypatch):
    B, S = 2, 32
    x = O.structured_batch(B, 0, T_CLIP, S)[0]
    x2 = O.structured_batch(B, 1, T_CLIP, S)[0]
    labels = torch.tensor([3, 77])
    a, b = _model(), _model()
    for m in (a, b):
        m.train()
        m.finetune_step(x, labels, lr=LR, momentum=MOM, weight_decay=WD)
    built = _count_builds(monkeypatch)
    bound = a._engine
    a.eval()
    evals = torch.rand(12, 3, T_CLIP, S, S, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        outs = {n: a(evals[:n], None, o_type="test") for n in range(1, 13)}
    assert sorted(built) == [("InferenceEngine", 1), ("InferenceEngine", 4), ("InferenceEngine", 8),
                             ("InferenceEngine", 16)]
    assert a._engine is bound and all(outs[n].shape == (n, 101) for n in outs)
    for n in range(1, 13):
        assert torch.allclose(outs[n], outs[12][:n], rtol=1e-5, atol=1e-6)
    a.train()
    b.train()
    la = a.finetune_step(x2, labels, lr=LR, momentum=MOM, weight_decay=WD)
    lb = b.finetune_step(x2, labels, lr=LR, momentum=MOM, weight_decay=WD)
    assert a._engine is bound and len(built) == 4
    assert torch.equal(la, lb)
    assert torch.equal(a._engine.mom, b._engine.mom) and torch.equal(a._engine.train.data, b._engine.train.data)
    assert torch.equal(a._engine.bufs.data, b._engine.bufs.data)
    a.free_inference_engines()
    assert not a._infer


def test_inference_engine_repacks_after_optimizer_step(emu):
    from cstp_b200 import engine_ft
    B, S = 2, 32
    x = O.structured_batch(B, 0, T_CLIP, S)[0]
    labels = torch.tensor([3, 77])
    m = _model()
    m.train()
    opt = torch.optim.SGD(m.parameters(), lr=LR, momentum=MOM, weight_decay=WD)
    ev = torch.rand(3, 3, T_CLIP, S, S, generator=torch.Generator().manual_seed(4))
    for step in range(2):
        loss = torch.nn.CrossEntropyLoss()(m(x, o_type="ft_all"), labels)
        opt.zero_grad()
        loss.backward()
        opt.step()
        m.eval()
        with torch.no_grad():
            got = m(ev, None, o_type="test")
            assert type(m._last_engine) is engine_ft.InferenceEngine and m._last_engine.capacity == 4
            ref = engine_ft.InferenceEngine(4, T_CLIP, S, S, device="cpu")       # packs the current weights afresh
            ref.train.data.copy_(m._engine.train.data)
            ref.bufs.data.copy_(m._engine.bufs.data)
            ref.pack_online()
            want = ref.forward_batch(ev)[:3, :101]
        assert torch.equal(got, want), step
        m.train()


def test_eval_first_owns_the_stores_until_a_training_engine_is_bound(emu):
    B, S = 2, 32
    m = _model()
    before = {k: v.clone() for k, v in m.state_dict().items()}
    m.eval()
    ev = torch.rand(3, 3, T_CLIP, S, S, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        first = m(ev, None, o_type="test")
    assert m._engine is None and m._infer_owner is not None
    assert m.online_net.conv1.spatial_conv.weight.data_ptr() == m._infer_owner.train.view(
        "online_net.conv1.spatial_conv.weight").data_ptr()
    m.train()
    m.finetune_step(O.structured_batch(B, 0, T_CLIP, S)[0], torch.tensor([1, 2]), lr=0.0, momentum=MOM, weight_decay=0.0)
    assert m._infer == {} and m._infer_owner is None
    assert m.online_net.conv1.spatial_conv.weight.data_ptr() == m._engine.train.view(
        "online_net.conv1.spatial_conv.weight").data_ptr()
    # lr 0: weights unchanged; the BatchNorm running statistics moved, so restore them and compare the eval logits
    m.load_state_dict(before)
    m.eval()
    with torch.no_grad():
        assert torch.equal(m(ev, None, o_type="test"), first)


# ------------------------------------------------------------------------------------------ world 2
def _worker_shard(rank, world, path, out):
    from cstp_b200 import engine
    from cstp_b200.evaluate import test_videos
    from tests import emulate_video_eval
    engine.ops, engine.ACT_DTYPE = emulate_video_eval, torch.float32
    dist.init_process_group("gloo", init_method=f"file://{path}", rank=rank, world_size=world)
    n = 5
    m = _model()
    m.eval()
    r = test_videos(m, _store(n), FRAMES[:n], [0, 1, 2, 3, 4], sample_duration=T_CLIP, capacity=3, rank=rank,
                    world=world, keep_logits=True, assemble=fake_assemble)
    torch.save(r, f"{out}.{rank}")
    dist.destroy_process_group()


def test_world2_shards_give_the_single_rank_counts(emu):
    from cstp_b200.evaluate import shard, test_videos
    d = tempfile.mkdtemp()
    path, out = os.path.join(d, "rdzv"), os.path.join(d, "out")
    mp.spawn(_worker_shard, args=(2, path, out), nprocs=2, join=True)
    r0, r1 = (torch.load(f"{out}.{r}", weights_only=False) for r in range(2))
    n = 5
    m = _model()
    m.eval()
    one = test_videos(m, _store(n), FRAMES[:n], [0, 1, 2, 3, 4], sample_duration=T_CLIP, capacity=3, keep_logits=True,
                      assemble=fake_assemble)
    assert list(shard(n, 0, 2)) == [0, 1] and list(shard(n, 1, 2)) == [2, 3, 4]
    for r in (r0, r1):
        assert (r["hits"], r["videos"], r["clips"], r["top1"], r["top5"]) == \
            (one["hits"], one["videos"], one["clips"], one["top1"], one["top5"])
    assert torch.equal(torch.cat([r0["predictions"], r1["predictions"]]), one["predictions"])
    assert torch.allclose(torch.cat([r0["logits"], r1["logits"]]), one["logits"], rtol=1e-5, atol=1e-6)   # CPU GEMM blocking


# ------------------------------------------------------------------------------------------ C ABI
def test_video_eval_entry_points_are_declared_and_bound():
    from cstp_b200 import lib as L
    header = (ROOT / "include" / "cstp_b200.h").read_text()
    for name in ("cstp_video_accumulate", "cstp_video_finalize"):
        assert re.search(rf"\bint {name}\(", header), name
        assert name in L.SIGNATURES
    if L.lib_path().exists():
        lib = L.load(build_if_missing=False)
        assert hasattr(lib, "cstp_video_accumulate") and hasattr(lib, "cstp_video_finalize")
