"""Monitoring a pretraining run, without a GPU: the float32 stand-in of cstp_repr_stats (tests/emulate_repr_stats.py)
against a float64 computation of the same definition, the wrapper's argument checks, and train.pretrain_epochs with
collapse_stats and a RetrievalMonitor over the emulated op layer (tests/emulate_retrieval.py plus the stand-in), on one
rank and on two."""
import os
import random
import tempfile
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import cstp_oracle as O
from tests import emulate_repr_stats as ER
from tests.test_video_eval_cpu import FRAMES, T_CLIP, _store, fake_assemble

LW = [0.1, 1.0, 1.0, 1.0, 1.0]


# ------------------------------------------------------------------------------------------ stand-in semantics
def _blocks(B, ld=512, seed=0, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(2 * B, ld, generator=g) * scale for _ in range(4)]


def _check_against_float64(blocks, B, got):
    for k, x in enumerate(blocks):
        ref = ER.float64_reference(x, B)
        for v in range(2):
            assert abs(got[v, k] - ref[v, 0]) <= 1e-5 * abs(ref[v, 0]), (k, v, got[v, k], ref[v, 0])
            if k == 0:
                assert abs(got[v, 4] - ref[v, 1]) <= 1e-5 * abs(ref[v, 1]), (v, got[v, 4], ref[v, 1])


@pytest.mark.parametrize("B", [2, 64])
def test_standin_matches_float64_on_random_rows(B):
    blocks = _blocks(B, seed=B, scale=0.3)
    blocks[1] = blocks[1] + 2.0               # rows far from the origin: the std is small against the mean
    got = ER.repr_stats_np(blocks, B)
    _check_against_float64(blocks, B, got)
    assert 0.02 < got[0, 0] < 0.07           # independent gaussian rows: about 1 / sqrt(512)


def test_standin_reads_only_512_columns_of_padded_rows():
    B, ld = 7, 528
    wide = _blocks(B, ld, seed=3)
    for x in wide:
        x[:, 512:] = float("nan")            # the padding is never read
    got = ER.repr_stats_np([x[:, :ld] for x in wide], B)
    assert np.isfinite(got).all()
    assert np.array_equal(got, ER.repr_stats_np([x[:, :512].contiguous() for x in wide], B))
    _check_against_float64([x[:, :512] for x in wide], B, got)


def test_identical_rows_give_exactly_zero():
    B = 60
    row = torch.randn(512, generator=torch.Generator().manual_seed(4))
    x = torch.cat([row.expand(B, 512), (3 * row).expand(B, 512)]).contiguous()     # each view constant
    got = ER.repr_stats_np([x, x, x, x], B)
    assert (got[:, :4] == 0).all()
    ref = ER.float64_reference(x, B)
    assert ref[:, 0].abs().max() < 1e-12
    assert abs(got[1, 4] / got[0, 4] - 3) < 1e-5


def test_all_zero_rows_go_through_the_clamp():
    B = 5
    x = torch.zeros(2 * B, 512)
    y = _blocks(B, seed=5)[0]
    y[B + 2] = 0                              # one zero row in view 2: z = 0 there, the others are unit rows
    got = ER.repr_stats_np([y, x, None, None], B)
    assert (got[:, 1:4] == 0).all()                         # all-zero rows: z = 0 / 1e-12; blocks not given: 0
    _check_against_float64([y], B, got)
    assert np.array_equal(ER.repr_stats_np([x, None, None, None], B)[:, [0, 4]], np.zeros((2, 2), np.float32))


def test_wrapper_rejects_bad_arguments_before_touching_a_device():
    from cstp_b200 import lib as L, ops
    B = 4
    x, out = torch.zeros(2 * B, 512), torch.zeros(2, 5)
    with pytest.raises(L.CstpError):
        ops.repr_stats(x[:2], x[:2], x[:2], x[:2], 1, out)                              # B < 2
    with pytest.raises(L.CstpError):
        ops.repr_stats(x.double(), x, x, x, B, out)                                     # not fp32
    with pytest.raises(L.CstpError):
        ops.repr_stats(x, x, x, x.bfloat16(), B, out)
    with pytest.raises(L.CstpError):
        ops.repr_stats(x, torch.zeros(2 * B, 256), x, x, B, out)                        # ld < 512
    with pytest.raises(L.CstpError):
        ops.repr_stats(x, x, torch.zeros(2 * B - 1, 512), x, B, out)                    # fewer than 2B rows
    with pytest.raises(L.CstpError):
        ops.repr_stats(x, x, x, x, B, torch.zeros(2, 5, dtype=torch.float64))
    with pytest.raises(L.CstpError):                                                    # valid arguments: the device check
        ops.repr_stats(x, x, x, x, B, out)


def test_entry_point_is_declared_and_bound():
    import re
    from pathlib import Path
    from cstp_b200 import lib as L
    header = (Path(__file__).resolve().parents[1] / "include" / "cstp_b200.h").read_text()
    assert re.search(r"\bint cstp_repr_stats\(", header) and "cstp_repr_stats" in L.SIGNATURES
    if L.lib_path().exists():
        assert hasattr(L.load(build_if_missing=False), "cstp_repr_stats")


# ------------------------------------------------------------------------------------------ the driver, emulated
N_GAL, N_QRY = 5, 3
GAL_LABELS, QRY_LABELS = [0, 1, 2, 0, 1], [0, 1, 2]
KS = (1, 2, 5)


def _opts(n_epochs):
    return types.SimpleNamespace(n_epochs=n_epochs, learning_rate=0.03, momentum=0.9, weight_decay=5e-4, clip_grad_norm=1,
                                 loss_weight=LW)


def _batches(epoch):
    for s in range(2):
        yield O.structured_batch(2, 10 * epoch + s, T_CLIP, 32)


def _model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    return R21DBYOL(pretrain=True)


def _monitor():
    from cstp_b200.train import RetrievalMonitor
    return RetrievalMonitor((_store(N_GAL), FRAMES[:N_GAL], GAL_LABELS), (_store(N_QRY), FRAMES[:N_QRY], QRY_LABELS),
                            ks=KS, sample_duration=T_CLIP, capacity=4, assemble=fake_assemble)


def _install():
    """engine.ops -> the emulated layer with the retrieval and repr_stats stand-ins; returns (restore, recorded stats)."""
    from cstp_b200 import engine
    from tests import emulate_ops, emulate_retrieval
    saved = engine.ops, engine.ACT_DTYPE, getattr(emulate_ops, "repr_stats", None)
    recorded = []

    def recording(feat, proj, pred, tproj, B, out):
        ER.repr_stats(feat, proj, pred, tproj, B, out)
        recorded.append(out.clone())
    engine.ops, engine.ACT_DTYPE = emulate_retrieval, torch.float32
    emulate_ops.repr_stats = recording

    def restore():
        engine.ops, engine.ACT_DTYPE = saved[0], saved[1]
        if saved[2] is None:
            del emulate_ops.repr_stats
        else:
            emulate_ops.repr_stats = saved[2]
    return restore, recorded


@pytest.fixture(scope="module")
def runs():
    """The same 3-epoch run twice: plain, and with collapse_stats plus a monitor every 2 epochs."""
    from cstp_b200 import train as TR
    restore, recorded = _install()
    try:
        d = tempfile.mkdtemp()
        plain_dir, mon_dir = os.path.join(d, "plain"), os.path.join(d, "mon")
        os.makedirs(plain_dir)
        os.makedirs(mon_dir)
        a = _model()
        rows_a = TR.pretrain_epochs(a, _batches, _opts(3), result_path=plain_dir, save_every=2)
        launches_a = list(recorded)
        b = _model()
        mon = _monitor()
        rows_b = TR.pretrain_epochs(b, _batches, _opts(3), result_path=mon_dir, save_every=2, collapse_stats=True,
                                    monitor=mon, monitor_every=2)
        stats = [s.clone() for s in recorded]
        from cstp_b200.evaluate import retrieve_videos, video_features
        g = video_features(b, _store(N_GAL), FRAMES[:N_GAL], sample_duration=T_CLIP, capacity=4, assemble=fake_assemble)
        q = video_features(b, _store(N_QRY), FRAMES[:N_QRY], sample_duration=T_CLIP, capacity=2, assemble=fake_assemble)
        direct = retrieve_videos(q, QRY_LABELS, g, GAL_LABELS, ks=KS)
        # generator states around one more evaluation
        random.seed(11)
        np.random.seed(11)
        torch.manual_seed(11)
        before = (random.getstate(), np.random.get_state(), torch.get_rng_state())
        again = mon(b)
        after = (random.getstate(), np.random.get_state(), torch.get_rng_state())
        yield dict(a=a, b=b, rows_a=rows_a, rows_b=rows_b, launches_a=launches_a, stats=stats, direct=direct,
                   again=again, before=before, after=after, plain_dir=plain_dir, mon_dir=mon_dir, g=g, q=q)
    finally:
        restore()


def test_nothing_requested_gives_todays_columns(runs):
    from cstp_b200.train import LOG_COLUMNS
    assert [list(r) for r in runs["rows_a"]] == [LOG_COLUMNS] * 3
    assert runs["launches_a"] == []                        # no statistics launch without collapse_stats


def test_monitoring_leaves_training_bit_identical(runs):
    from cstp_b200.train import LOG_COLUMNS
    for ra, rb in zip(runs["rows_a"], runs["rows_b"]):
        assert [rb[c] for c in LOG_COLUMNS] == [ra[c] for c in LOG_COLUMNS]
    sa, sb = runs["a"].state_dict(), runs["b"].state_dict()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    assert torch.equal(runs["a"]._engine.mom, runs["b"]._engine.mom)
    assert sorted(os.listdir(runs["plain_dir"])) == sorted(os.listdir(runs["mon_dir"])) == ["save_2.pth", "save_3.pth"]
    for f in ("save_2.pth", "save_3.pth"):
        ca = torch.load(os.path.join(runs["plain_dir"], f), weights_only=False)
        cb = torch.load(os.path.join(runs["mon_dir"], f), weights_only=False)
        assert ca["state_dict"].keys() == cb["state_dict"].keys()
        assert all(torch.equal(ca["state_dict"][k], cb["state_dict"][k]) for k in ca["state_dict"])
        assert all(torch.equal(ca["optimizer"]["state"][i]["momentum_buffer"], cb["optimizer"]["state"][i]["momentum_buffer"])
                   for i in ca["optimizer"]["state"])


def test_collapse_columns_are_the_epoch_mean_of_the_step_statistics(runs):
    from cstp_b200.ops import REPR_STATS
    stats = runs["stats"]
    assert len(stats) == 6                                  # one launch per step, 2 steps x 3 epochs
    for e, row in enumerate(runs["rows_b"]):
        S = torch.stack(stats[2 * e:2 * e + 2]).mean(0)
        for i, name in enumerate(REPR_STATS):
            assert row[name] == ((S[0, i] + S[1, i]) / 2).item(), (e, name)
        assert 0 < row["std_feat"] < 1 and row["feat_norm"] > 0


def test_monitor_epochs_and_recall_columns(runs):
    rec = [f"recall@{k}" for k in KS]
    assert [all(c in r for c in rec) for r in runs["rows_b"]] == [False, True, True]     # every 2nd epoch and the last
    last = runs["rows_b"][-1]
    assert [last[c] for c in rec] == [runs["direct"]["recall"][k] for k in KS]
    assert runs["again"] == {c: last[c] for c in rec}
    assert runs["g"].shape == (N_GAL, 512) and (runs["g"].norm(dim=1) > 0).all()


def test_evaluation_draws_nothing_from_the_generators(runs):
    b, a = runs["before"], runs["after"]
    assert b[0] == a[0]
    assert all(np.array_equal(x, y) if isinstance(x, np.ndarray) else x == y for x, y in zip(b[1], a[1]))
    assert torch.equal(b[2], a[2])


def test_test_windows_are_deterministic():
    """plan_test is a function of (frames, size): the monitor's clips are the same at every evaluation."""
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    random.seed(1)
    s1 = FinetuneClipSampler(16, 112, 4)
    p1 = [s1.plan_test(n, 171, 128) for n in (29, 61, 200, 1800)]
    random.seed(2)
    np.random.seed(2)
    torch.manual_seed(2)
    s2 = FinetuneClipSampler(16, 112, 4)
    p2 = [s2.plan_test(n, 171, 128) for n in (29, 61, 200, 1800)]
    assert [[(c.view.frames, c.view.box) for c in p] for p in p1] == [[(c.view.frames, c.view.box) for c in p] for p in p2]


def test_feature_extraction_needs_a_bound_step_engine():
    from cstp_b200 import lib as L
    from cstp_b200.evaluate import video_features
    with pytest.raises(L.CstpError):
        video_features(_model(), _store(1), FRAMES[:1], sample_duration=T_CLIP, assemble=fake_assemble)


def test_monitor_rejects_bad_arguments():
    from cstp_b200.train import RetrievalMonitor, pretrain_epochs
    side = (_store(2), FRAMES[:2], [0, 1])
    for ks in ((0,), (65,), ()):
        with pytest.raises(ValueError):
            RetrievalMonitor(side, side, ks=ks)
    with pytest.raises(ValueError):
        RetrievalMonitor(side, (side[0], FRAMES[:2], [0]))
    with pytest.raises(ValueError):
        pretrain_epochs(_model(), _batches, _opts(1), monitor_every=0)


# ------------------------------------------------------------------------------------------ world 2
def _worker(rank, world, path, out):
    from cstp_b200 import parallel as P, train as TR
    from cstp_b200.evaluate import retrieve_videos, video_features
    torch.set_num_threads(2)
    _, recorded = _install()
    dist.init_process_group("gloo", init_method=f"file://{path}", rank=rank, world_size=world)
    lo, hi = P.shard_bounds(4, rank, world)

    def batches(epoch):
        for s in range(2):
            x1, x2, lab = O.structured_batch(4, 10 * epoch + s, T_CLIP, 32)
            yield x1[lo:hi].contiguous(), x2[lo:hi].contiguous(), tuple(l[lo:hi].contiguous() for l in lab)
    m = _model()
    rows = TR.pretrain_epochs(m, batches, _opts(2), grad_sync=P.GradSync(), collapse_stats=True, monitor=_monitor(),
                              monitor_every=5)
    g = video_features(m, _store(N_GAL), FRAMES[:N_GAL], sample_duration=T_CLIP, capacity=4, assemble=fake_assemble)
    q = video_features(m, _store(N_QRY), FRAMES[:N_QRY], sample_duration=T_CLIP, capacity=4, assemble=fake_assemble)
    local = retrieve_videos(q, QRY_LABELS, g, GAL_LABELS, ks=KS)["recall"]
    torch.save({"rows": rows, "stats": [s.clone() for s in recorded], "local": local}, f"{out}.{rank}")
    dist.destroy_process_group()


def test_world2_rows_average_the_ranks():
    from cstp_b200.ops import REPR_STATS
    d = tempfile.mkdtemp()
    path, out = os.path.join(d, "rdzv"), os.path.join(d, "out")
    mp.spawn(_worker, args=(2, path, out), nprocs=2, join=True)
    r0, r1 = (torch.load(f"{out}.{r}", weights_only=False) for r in range(2))
    assert r0["rows"] == r1["rows"]                         # every rank logs the same row
    for e, row in enumerate(r0["rows"]):
        S = (torch.stack(r0["stats"][2 * e:2 * e + 2]).mean(0) + torch.stack(r1["stats"][2 * e:2 * e + 2]).mean(0)) / 2
        for i, name in enumerate(REPR_STATS):
            assert row[name] == pytest.approx(((S[0, i] + S[1, i]) / 2).item(), rel=1e-6), (e, name)
    assert "recall@1" not in r0["rows"][0]                  # monitor_every 5: only the last epoch is evaluated
    last = r0["rows"][-1]
    assert [last[f"recall@{k}"] for k in KS] == [r0["local"][k] for k in KS] == [r1["local"][k] for k in KS]
