"""Nearest-neighbour video retrieval on CPU: the float32 stand-ins of cstp_l2_normalize_rows / cstp_knn_partial /
cstp_knn_merge (tests/emulate_retrieval.py) against a float64 brute force, their total order (ties, k > gallery, cutoffs
past the gallery), and cstp_b200.evaluate.video_features / retrieve_videos over the CPU emulator, on one rank and two."""
import os
import tempfile

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.test_video_eval_cpu import FRAMES, T_CLIP, _model, _store, fake_assemble, seq_mean


@pytest.fixture()
def emu():
    from cstp_b200 import engine
    from tests import emulate_retrieval
    saved = engine.ops, engine.ACT_DTYPE
    engine.ops, engine.ACT_DTYPE = emulate_retrieval, torch.float32
    try:
        yield engine
    finally:
        engine.ops, engine.ACT_DTYPE = saved


def _search(q, g, k, splits, ql=None, gl=None, cutoffs=None):
    """The three stand-ins in the order retrieve_videos launches them."""
    from tests import emulate_retrieval as E
    qn, gn = torch.empty_like(q), torch.empty_like(g)
    E.l2_normalize_rows(q, qn)
    E.l2_normalize_rows(g, gn)
    pv = torch.empty(splits, q.shape[0], k)
    pi = torch.empty(splits, q.shape[0], k, dtype=torch.int32)
    E.knn_partial(qn, gn, k, splits, pv, pi)
    idx = torch.empty(q.shape[0], k, dtype=torch.int64)
    sim = torch.empty(q.shape[0], k)
    hits = None if cutoffs is None else torch.zeros(len(cutoffs), dtype=torch.int64)
    E.knn_merge(pv, pi, idx, sim, ql, gl, None if cutoffs is None else torch.tensor(cutoffs, dtype=torch.int32), hits)
    return idx, sim, hits


def test_normalize_standin_is_f_normalize():
    from tests import emulate_retrieval as E
    x = torch.randn(9, 100, generator=torch.Generator().manual_seed(1))
    x[3] = 0
    y = torch.empty(9, 100)
    E.l2_normalize_rows(x, y)
    assert torch.allclose(y, torch.nn.functional.normalize(x, dim=1), rtol=1e-6, atol=1e-7)
    assert not y[3].any()


@pytest.mark.parametrize("k", [1, 10, 50])
def test_standin_matches_float64_brute_force(emu, k):
    from cstp_b200.evaluate import retrieve_videos
    g = torch.Generator().manual_seed(k)
    q, gal = torch.randn(40, 64, generator=g), torch.randn(300, 64, generator=g)
    ql, gl = torch.randint(0, 7, (40,), generator=g), torch.randint(0, 7, (300,), generator=g)
    ks = sorted({1, 5, k})
    r = retrieve_videos(q, ql, gal, gl, ks=ks)
    s64 = torch.nn.functional.normalize(q.double(), dim=1) @ torch.nn.functional.normalize(gal.double(), dim=1).T
    ref = torch.sort(s64, dim=1, descending=True)
    checked = 0
    for i in range(40):
        if ref.values[i, k - 1] - ref.values[i, k] <= 1e-6:
            continue
        checked += 1
        assert set(r["neighbours"][i, :k].tolist()) == set(ref.indices[i, :k].tolist()), i
    assert checked >= 35
    assert torch.allclose(r["similarity"][:, :k].double(), ref.values[:, :k], atol=1e-6)
    for c in ks:
        want = sum(int((gl[ref.indices[i, :c]] == ql[i]).any()) for i in range(40))
        assert r["hits"][c] == want and r["recall"][c] == want / 40
    assert r["queries"] == 40 and r["neighbours"].shape == (40, max(ks))


def test_ties_go_to_the_lower_gallery_index_for_every_split():
    g = torch.Generator().manual_seed(3)
    base = torch.randn(5, 16, generator=g)
    gal = torch.cat([base, base, 2 * base[:2]])             # rows i, i + 5 (and 10, 11 scaled) tie exactly
    q = base[[1, 3]] + 0.01 * torch.randn(2, 16, generator=g)
    runs = [_search(q, gal, 12, s)[:2] for s in (1, 2, 5)]
    for idx, sim in runs[1:]:
        assert torch.equal(idx, runs[0][0]) and torch.equal(sim, runs[0][1])
    idx, sim = runs[0]
    assert idx[0, :3].tolist() == [1, 6, 11] and sim[0, 0] == sim[0, 1] == sim[0, 2]
    assert idx[1, :2].tolist() == [3, 8]
    for r in range(2):                                      # non-increasing, and ascending index on equal values
        for j in range(11):
            assert sim[r, j] > sim[r, j + 1] or (sim[r, j] == sim[r, j + 1] and idx[r, j] < idx[r, j + 1])


def test_zero_rows_score_zero_and_rank_by_index():
    q = torch.zeros(1, 8)
    gal = torch.randn(6, 8, generator=torch.Generator().manual_seed(2))
    idx, sim, _ = _search(q, gal, 6, 2)
    assert idx[0].tolist() == list(range(6)) and not sim.any()


def test_k_beyond_the_gallery_pads_with_minus_one_and_minus_inf():
    g = torch.Generator().manual_seed(4)
    q, gal = torch.randn(3, 8, generator=g), torch.randn(4, 8, generator=g)
    idx, sim, _ = _search(q, gal, 7, 3)
    assert (idx[:, 4:] == -1).all() and torch.isneginf(sim[:, 4:]).all()
    assert sorted(idx[0, :4].tolist()) == [0, 1, 2, 3] and torch.isfinite(sim[:, :4]).all()


def test_cutoffs_beyond_the_gallery_count_the_whole_gallery(emu):
    from cstp_b200.evaluate import retrieve_videos
    g = torch.Generator().manual_seed(5)
    q, gal = torch.randn(6, 8, generator=g), torch.randn(4, 8, generator=g)
    ql = torch.tensor([0, 1, 2, 3, 9, 9])
    gl = torch.tensor([3, 2, 1, 0])
    r = retrieve_videos(q, ql, gal, gl, ks=(1, 4, 5, 10))
    assert r["hits"][4] == r["hits"][5] == r["hits"][10] == 4 and r["recall"][10] == 4 / 6
    assert (r["neighbours"][:, 4:] == -1).all()


def test_retrieve_videos_rejects_cutoffs_outside_1_to_64(emu):
    from cstp_b200.evaluate import retrieve_videos
    x = torch.randn(2, 8)
    for ks in ((0, 5), (1, 65), ()):
        with pytest.raises(ValueError):
            retrieve_videos(x, [0, 1], x, [0, 1], ks=ks)
    with pytest.raises(ValueError):
        retrieve_videos(torch.randn(2, 6), [0, 1], torch.randn(2, 6), [0, 1])


@pytest.mark.parametrize("case", ["bf16_query", "fp16_gallery", "fp64_query", "1d_gallery", "short_gallery_labels",
                                  "long_gallery_labels", "short_query_labels", "nested_query_labels"])
def test_retrieve_videos_rejects_features_and_labels_that_do_not_match(emu, case):
    """The kernels read fp32 rows and index the labels by row: anything else must fail on the host, never on the device."""
    from cstp_b200.evaluate import retrieve_videos
    q, g = torch.randn(5, 8), torch.randn(7, 8)
    ql, gl = list(range(5)), list(range(7))
    args = {"bf16_query": (q.bfloat16(), ql, g, gl), "fp16_gallery": (q, ql, g.half(), gl),
            "fp64_query": (q.double(), ql, g, gl), "1d_gallery": (q, ql, g[0], gl),
            "short_gallery_labels": (q, ql, g, gl[:6]), "long_gallery_labels": (q, ql, g, gl + [0]),
            "short_query_labels": (q, ql[:4], g, gl), "nested_query_labels": (q, [ql], g, gl)}[case]
    with pytest.raises(ValueError):
        retrieve_videos(*args, ks=(1, 5))
    assert retrieve_videos(q, torch.tensor(ql), g, torch.tensor(gl), ks=(1, 5))["queries"] == 5


# ------------------------------------------------------------------------------------------ video_features
def per_video_feature_means(m, store, n, T, S, device, plans_of, assemble):
    """Today's path for one video at a time: FinetuneEngine(clips).forward_eval on the module's current weights, then the
    sequential fp32 mean of the pooled feature rows."""
    from cstp_b200 import engine_ft
    src = m._engine if m._engine is not None else m._infer_owner
    means = []
    with torch.no_grad():
        for v in range(n):
            plans = plans_of(v)
            x = assemble(plans, [store[v]] * len(plans), torch.empty(len(plans), 3, T, S, S, device=device))
            ref = engine_ft.FinetuneEngine(len(plans), T, S, S, device=device, **getattr(m, "engine_options", {}))
            ref.train.data.copy_(src.train.data)
            ref.bufs.data.copy_(src.bufs.data)
            ref.pack_online()
            ref.forward_eval(x)
            means.append(seq_mean(ref.feat[:len(plans)].cpu()))
    return torch.stack(means)


def test_video_features_equal_per_video_forward_eval_means(emu):
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    from cstp_b200.evaluate import video_features
    n = len(FRAMES)
    store = _store(n)
    m = _model()
    m.eval()
    f = video_features(m, store, FRAMES, sample_duration=T_CLIP, capacity=7, assemble=fake_assemble)
    sampler = FinetuneClipSampler(T_CLIP, 112, 4)
    ref = per_video_feature_means(m, store, n, T_CLIP, 112, "cpu", lambda v: sampler.plan_test(FRAMES[v], 12, 8),
                                  fake_assemble)
    assert f.shape == (n, 512) and f.dtype == torch.float32
    # the CPU stand-in's fp32 GEMMs block differently for different batch sizes (tests/test_gpu_retrieval.py compares bits)
    assert torch.allclose(f, ref, rtol=1e-5, atol=1e-6)
    assert (f.norm(dim=1) > 0).all()


# ------------------------------------------------------------------------------------------ world 2
N_W2 = 5


def _fixed_features():
    g = torch.Generator().manual_seed(8)
    return torch.randn(7, 32, generator=g), torch.randint(0, 3, (7,), generator=g), torch.randn(11, 32, generator=g), \
        torch.randint(0, 3, (11,), generator=g)


def _worker(rank, world, path, out):
    from cstp_b200 import engine
    from cstp_b200.evaluate import retrieve_videos, video_features
    from tests import emulate_retrieval
    engine.ops, engine.ACT_DTYPE = emulate_retrieval, torch.float32
    dist.init_process_group("gloo", init_method=f"file://{path}", rank=rank, world_size=world)
    m = _model()
    m.eval()
    f = video_features(m, _store(N_W2), FRAMES[:N_W2], sample_duration=T_CLIP, capacity=3, rank=rank, world=world,
                       assemble=fake_assemble)
    q, ql, g, gl = _fixed_features()
    r = retrieve_videos(q, ql, g, gl, ks=(1, 3, 5), rank=rank, world=world)
    torch.save({"features": f, "retrieval": r}, f"{out}.{rank}")
    dist.destroy_process_group()


def test_world2_gives_the_single_rank_features_and_hits(emu):
    from cstp_b200.evaluate import retrieve_videos, shard, video_features
    d = tempfile.mkdtemp()
    path, out = os.path.join(d, "rdzv"), os.path.join(d, "out")
    mp.spawn(_worker, args=(2, path, out), nprocs=2, join=True)
    r0, r1 = (torch.load(f"{out}.{r}", weights_only=False) for r in range(2))
    m = _model()
    m.eval()
    one = video_features(m, _store(N_W2), FRAMES[:N_W2], sample_duration=T_CLIP, capacity=3, assemble=fake_assemble)
    q, ql, g, gl = _fixed_features()
    ref = retrieve_videos(q, ql, g, gl, ks=(1, 3, 5))
    for r in (r0, r1):
        assert r["features"].shape == one.shape
        assert torch.allclose(r["features"], one, rtol=1e-5, atol=1e-6)          # CPU GEMM blocking
        assert r["retrieval"]["hits"] == ref["hits"] and r["retrieval"]["recall"] == ref["recall"]
        assert r["retrieval"]["queries"] == 7
    assert torch.equal(r0["features"], r1["features"])
    assert len(shard(7, 0, 2)) == 3 and len(shard(7, 1, 2)) == 4
    assert torch.equal(torch.cat([r0["retrieval"]["neighbours"], r1["retrieval"]["neighbours"]]), ref["neighbours"])
    assert torch.equal(torch.cat([r0["retrieval"]["similarity"], r1["retrieval"]["similarity"]]), ref["similarity"])


# ------------------------------------------------------------------------------------------ C ABI
def test_retrieval_entry_points_are_declared_and_bound():
    import re
    from pathlib import Path
    from cstp_b200 import build, lib as L
    header = (Path(__file__).resolve().parents[1] / "include" / "cstp_b200.h").read_text()
    for name in ("cstp_l2_normalize_rows", "cstp_knn_partial", "cstp_knn_merge"):
        assert re.search(rf"\bint {name}\(", header), name
        assert name in L.SIGNATURES
    assert "retrieval.cu" in build.SOURCES
    if L.lib_path().exists():
        lib = L.load(build_if_missing=False)
        assert all(hasattr(lib, n) for n in ("cstp_l2_normalize_rows", "cstp_knn_partial", "cstp_knn_merge"))


def test_host_split_choice_stays_within_the_kernel_limits():
    from cstp_b200 import ops
    for nq, ng in [(1, 1), (300, 1237), (3783, 9537), (19715, 239429), (1, 10 ** 6), (10 ** 5, 600)]:
        s = ops.knn_splits(nq, ng)
        assert 1 <= s <= ops.KNN_MAX_SPLITS and (s == 1 or ng // s >= 512)
