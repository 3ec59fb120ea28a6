"""Video-level test evaluation on the B200: the clip-averaging / top-k kernels against sequential fp32 and torch.topk,
the padded-capacity inference engine against an exact-batch FinetuneEngine (bit-identical logits), and
cstp_b200.evaluate.test_videos end to end against the drop-in per-video loop of test.py:76-93 and the CPU oracle."""
import pytest
import torch

from tests.parity import rel

pytestmark = pytest.mark.gpu
LR, MOM, WD = 0.025, 0.9, 1e-3


def _model(**options):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
    m.engine_options = dict(options)
    return m.cuda()


def seq_sum(rows):
    acc = rows[0].clone()
    for r in rows[1:]:
        acc += r
    return acc


# ------------------------------------------------------------------------------------------ kernels
def test_accumulate_finalize_kernels_against_sequential_fp32_and_topk():
    from cstp_b200 import ops
    from cstp_b200.evaluate import batch_tables
    g = torch.Generator().manual_seed(7)
    counts = [int(c) for c in torch.randint(1, 41, (150,), generator=g)] + [1, 1, 40]
    V, C, cap, k = len(counts), 101, 60, 8
    logits = torch.randn(sum(counts), 112, generator=g)
    labels = torch.randint(0, C, (V,), generator=g)
    tab = torch.from_numpy(batch_tables(counts, cap)).cuda()
    sums = torch.zeros(V, C, device="cuda")
    mean = torch.zeros(V, C, device="cuda")
    topk = torch.zeros(V, k, dtype=torch.int64, device="cuda")
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    buf = torch.full((cap, 112), float("nan"), device="cuda")              # padding rows must never be read
    labels_dev = labels.cuda()
    table = torch.zeros_like(tab[0])                # all-zero work lists: every entry is skipped

    def launches():
        ops.video_accumulate(buf, C, table[0], sums)
        ops.video_finalize(sums, table[1], topk, labels_dev, mean, hits)
    launches()                                      # eager warm-up
    torch.cuda.synchronize()
    # one CUDA graph: the input rows and the work lists are rewritten in place before every replay
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        launches()
    for b in range(tab.shape[0]):
        rows = logits[b * cap:(b + 1) * cap]
        buf.fill_(float("nan"))
        buf[:rows.shape[0]].copy_(rows)
        table.copy_(tab[b])
        graph.replay()
    torch.cuda.synchronize()
    assert not sums.any()
    mean, topk, hits = mean.cpu(), topk.cpu(), hits.cpu()
    start, h1, h5 = 0, 0, 0
    for v, n in enumerate(counts):
        rows = logits[start:start + n, :C]
        start += n
        ref = seq_sum(rows) / float(n)
        assert torch.equal(mean[v], ref), v
        assert topk[v].tolist() == torch.topk(ref, k).indices.tolist(), v                 # no ties in random data
        h1 += int(topk[v, 0] == labels[v])
        h5 += int(labels[v] in topk[v, :5].tolist())
    assert hits.tolist() == [h1, h5]


def test_finalize_ties_go_to_the_lower_class_index():
    from cstp_b200 import ops
    x = torch.zeros(1, 256, device="cuda")
    x[0, [200, 7, 130, 3]] = 1.5
    x[0, [99, 11]] = 0.25
    sums = torch.zeros(1, 250, device="cuda")
    topk = torch.zeros(1, 8, dtype=torch.int64, device="cuda")
    hits = torch.zeros(2, dtype=torch.int64, device="cuda")
    ops.video_accumulate(x, 250, torch.tensor([[0, 0, 1]], dtype=torch.int32, device="cuda"), sums)
    ops.video_finalize(sums, torch.tensor([[0, 1, 0]], dtype=torch.int32, device="cuda"), topk,
                       torch.tensor([99], device="cuda"), None, hits)
    assert topk.cpu().tolist() == [[3, 7, 130, 200, 11, 99, 0, 1]] and hits.cpu().tolist() == [0, 0]


# ------------------------------------------------------------------------------------------ inference engine
def _reference_logits(m, x, T, S):
    """Today's path for exactly this batch: FinetuneEngine(n).forward_eval on the module's current weights."""
    from cstp_b200 import engine_ft
    ref = engine_ft.FinetuneEngine(x.shape[0], T, S, S, device="cuda", **m.engine_options)
    ref.train.data.copy_(m._engine.train.data)
    ref.bufs.data.copy_(m._engine.bufs.data)
    ref.pack_online()
    return ref.forward_eval(x)[:, :101].clone()


@pytest.mark.parametrize("T,S,options", [(8, 64, {}), (8, 64, {"fuse_min_positions": 0}), (16, 112, {})])
def test_padded_capacity_engine_is_bit_identical_to_exact_batch(T, S, options):
    from oracle import cstp_oracle as O
    from cstp_b200 import engine_ft
    m = _model(**options).train()
    x = O.structured_batch(2, 0, T, S)[0].cuda()
    labels = torch.tensor([3, 77], device="cuda")
    m.finetune_step(x, labels, lr=LR, momentum=MOM, weight_decay=WD)
    ev = (torch.rand(33, 3, T, S, S, generator=torch.Generator().manual_seed(2)) * 2 - 1).cuda()
    ns = (1, 3, 7, 33) if S == 64 else (3, 7)
    for step in range(2):
        m.eval()
        with torch.no_grad():
            for n in ns:
                got = m(ev[:n], None, o_type="test")
                eng = m._last_engine
                assert type(eng) is engine_ft.InferenceEngine and eng.capacity == engine_ft.inference_capacity(n)
                assert torch.equal(got, _reference_logits(m, ev[:n], T, S)), (step, n)
        m.train()
        m.finetune_step(x, labels, lr=LR, momentum=MOM, weight_decay=WD)        # the engines must re-pack


# ------------------------------------------------------------------------------------------ test_videos
FRAMES = [29, 95, 200, 61, 130, 45, 64, 250]


def _synthetic_store(n):
    from cstp_b200.data_process.datasets import GpuVideoStore
    store = GpuVideoStore()
    g = torch.Generator().manual_seed(9)
    for v in range(n):
        store.put(v, torch.randint(0, 256, (FRAMES[v], 128, 171, 3), dtype=torch.uint8, generator=g))
    return store


def test_test_videos_end_to_end(monkeypatch):
    from oracle import cstp_oracle as O
    from cstp_b200 import engine_ft
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    from cstp_b200.data_process.gpu_clips import GpuClipPipeline
    from cstp_b200.evaluate import test_videos
    n = len(FRAMES)
    store = _synthetic_store(n)
    m = _model().train()
    x = O.structured_batch(2, 0, 16, 112)[0].cuda()
    m.finetune_step(x, torch.tensor([3, 77], device="cuda"), lr=LR, momentum=MOM, weight_decay=WD)
    built = []
    init = engine_ft.InferenceEngine.__init__

    def spy(self, capacity, *a, **k):
        built.append(capacity)
        init(self, capacity, *a, **k)
    monkeypatch.setattr(engine_ft.InferenceEngine, "__init__", spy)
    # ---- the drop-in per-video loop of test.py:76-93
    m.eval()
    sampler, pipe = FinetuneClipSampler(16, 112, 4), GpuClipPipeline(16, 112)
    means, clips_of = [], []
    with torch.no_grad():
        for v in range(n):
            plans = sampler.plan_test(FRAMES[v], 171, 128)
            clips = pipe.assemble_clips(plans, [store[v]] * len(plans))
            # on the host: torch's CUDA division by a scalar multiplies by its reciprocal, the kernel divides
            means.append(seq_sum(m(clips, None, o_type="test").cpu()) / float(len(plans)))
            clips_of.append(clips)
    counts = [c.shape[0] for c in clips_of]
    assert len(set(counts)) >= 3
    buckets = {engine_ft.inference_capacity(c) for c in counts if c != 2}     # batch 2 is the bound engine's own
    assert sorted(built) == sorted(buckets)                                   # one engine per bucket, none per video
    ref = torch.stack(means)
    labels = torch.randint(0, 101, (n,), generator=torch.Generator().manual_seed(4))
    labels[:3] = ref[:3].argmax(1)                                           # a few hits
    top = torch.topk(ref, 5).indices
    want = ((top[:, 0] == labels).sum().item(), (top == labels[:, None]).any(1).sum().item())
    # ---- packed: capacity 3, so most videos straddle batches
    runs = [test_videos(m, store, FRAMES, labels.tolist(), capacity=3, keep_logits=True) for _ in range(2)]
    r = runs[0]
    assert built[-1] == 3 and len(built) == len(buckets) + 1
    assert torch.equal(r["logits"], ref)
    assert torch.equal(r["predictions"], top)
    assert r["hits"] == want and r["top1"] == want[0] / n and r["top5"] == want[1] / n and want[0] >= 3
    assert r["videos"] == n and r["clips"] == sum(counts)
    assert torch.equal(runs[1]["logits"], r["logits"]) and torch.equal(runs[1]["predictions"], r["predictions"])
    # ---- the CPU oracle on two clips, within the eval bound of tests/test_gpu_finetune.py
    state = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    clip = torch.cat([clips_of[0][:1], clips_of[2][1:2]]).cpu()
    with torch.no_grad():
        want_logits, _ = O.finetune_forward(state, clip, training=False)
        got = m(clip.cuda(), None, o_type="test").cpu()
    assert rel(got, want_logits) < 0.1
