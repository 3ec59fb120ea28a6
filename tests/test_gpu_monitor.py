"""Monitoring a pretraining run on the B200: cstp_repr_stats bit-exact against its float32 stand-in
(tests/emulate_repr_stats.py) on the engine's own buffers, in the captured step and eagerly; a step with collapse_stats
leaving every training buffer bit-identical; the features of the live pretraining model bit-identical to those of the
finetune model loaded from its checkpoint, from a store and from JPEG frames; and the epoch driver with a monitor."""
import os
import tempfile
import types

import pytest
import torch
from PIL import features

from tests import emulate_repr_stats as ER

pytestmark = pytest.mark.gpu
LW = (0.1, 1.0, 1.0, 1.0, 1.0)


def _model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(0)
    return R21DBYOL(pretrain=True).cuda().train()


def _batch(B, T=16, S=112, seed=2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    x1 = torch.rand(B, 3, T, S, S, device="cuda", generator=g) * 2 - 1
    x2 = torch.rand(B, 3, T, S, S, device="cuda", generator=g) * 2 - 1
    labels = tuple(torch.randint(0, 5, (B,), device="cuda", generator=g) for _ in range(5))
    return x1, x2, labels


def _standin(eng):
    return torch.from_numpy(ER.repr_stats_np([eng.feat, eng.proj_out, eng.pred, eng.tproj], eng.B))


def _state(m):
    eng = m._engine
    return {"losses": eng.losses.clone(), "train": eng.train.data.clone(), "grad": eng.grad.clone(),
            "mom": eng.mom.clone(), "bufs": eng.bufs.data.clone(), "target": eng.target.data.clone(),
            "nbt": m._nbt.clone()}


# ------------------------------------------------------------------------------------------ kernel and engine
@pytest.fixture(scope="module")
def b60():
    """Two batch-60 models from the same weights, three steps each on the same clips (eager, captured, replayed): one
    with collapse_stats, one without.  Records the statistics and every training buffer after each step."""
    from cstp_b200 import ops
    x1, x2, labels = _batch(60)
    out = {}
    for on in (False, True):
        m = _model()
        rec = []
        for step in range(3):
            n0 = ops.launch_count()
            m.train_step(x1, x2, labels, LW, lr=0.03, collapse_stats=on)
            torch.cuda.synchronize()
            launches = ops.launch_count() - n0
            eng = m._engine
            rec.append(dict(_state(m), launches=launches, graph=eng._graph is not None,
                            stats=m.step_stats().clone() if on else None, standin=_standin(eng) if on else None))
        out[on] = (m, rec)
    return out


def test_kernel_is_bit_exact_against_the_standin_on_the_engine_buffers(b60):
    from cstp_b200 import ops
    m, rec = b60[True]
    assert [r["graph"] for r in rec] == [False, True, True]
    for r in rec:                                        # eager step, capture step, replayed step
        assert torch.equal(r["stats"].cpu(), r["standin"]), r["stats"]
    eng = m._engine
    again = [torch.zeros(2, 5, device="cuda") for _ in range(2)]
    for o in again:                                      # eager launches on the replayed step's buffers
        ops.repr_stats(eng.feat, eng.proj_out, eng.pred, eng.tproj, eng.B, o)
    torch.cuda.synchronize()
    assert torch.equal(again[0], again[1]) and torch.equal(again[0].cpu(), rec[-1]["stats"].cpu())
    s = rec[0]["stats"].cpu()
    assert torch.isfinite(s).all() and (s[:, :4] > 0).all() and (s[:, 4] > 0).all()


def test_statistics_leave_every_training_buffer_bit_identical(b60):
    _, off = b60[False]
    _, on = b60[True]
    for step, (a, b) in enumerate(zip(off, on)):
        for k in ("losses", "train", "grad", "mom", "bufs", "target", "nbt"):
            assert torch.equal(a[k], b[k]), (step, k)


def test_launch_count_is_one_higher_with_statistics(b60):
    _, off = b60[False]
    _, on = b60[True]
    assert [b["launches"] - a["launches"] for a, b in zip(off, on)] == [1, 1, 1]


def test_switching_the_setting_recaptures_the_step():
    m = _model()
    x1, x2, labels = _batch(4, 8, 64)
    for step, on in enumerate((False, False, True, True, False)):
        m.train_step(x1, x2, labels, LW, lr=0.03, collapse_stats=on)
        assert (m._engine._graph is not None) == (step > 0) and m._engine.collapse_stats == on
    ref = _model()
    for _ in range(5):
        ref.train_step(x1, x2, labels, LW, lr=0.03)
    torch.cuda.synchronize()
    assert torch.equal(ref._engine.train.data, m._engine.train.data)
    assert torch.equal(ref._engine.bufs.data, m._engine.bufs.data)


def test_wrapper_and_entry_point_reject_bad_arguments():
    import ctypes as C
    from cstp_b200 import lib as L, ops
    x, out = torch.zeros(8, 512, device="cuda"), torch.zeros(2, 5, device="cuda")
    for args in ((x[:2], None, None, None, 1, out), (x.half(), None, None, None, 4, out),
                 (torch.zeros(8, 256, device="cuda"), None, None, None, 4, out)):
        with pytest.raises(L.CstpError):
            ops.repr_stats(*args)
    lib = L.load()
    p = x.data_ptr()
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.cstp_repr_stats(C.c_void_p(p), 512, None, 0, None, 0, None, 0, 1, C.c_void_p(out.data_ptr()), s) == -1
    assert lib.cstp_repr_stats(C.c_void_p(p), 500, None, 0, None, 0, None, 0, 4, C.c_void_p(out.data_ptr()), s) == -1
    assert lib.cstp_repr_stats(C.c_void_p(p + 2), 512, None, 0, None, 0, None, 0, 4, C.c_void_p(out.data_ptr()), s) == -1
    ops.repr_stats(x, None, None, None, 4, out)                      # zeros in, zeros out
    torch.cuda.synchronize()
    assert not out.any()


def test_collapsed_batch_drives_the_std_to_zero():
    m = _model()
    x1, x2, labels = _batch(16)
    m.train_step(x1, x2, labels, LW, lr=0.03, collapse_stats=True)
    spread = m.step_stats().cpu()
    same1, same2 = x1[:1].expand_as(x1).contiguous(), x2[:1].expand_as(x2).contiguous()
    m.train_step(same1, same2, labels, LW, lr=0.03, collapse_stats=True)
    collapsed = m.step_stats().cpu()
    print(f"random batch {spread.tolist()}  collapsed batch {collapsed.tolist()}")
    assert (0.01 < spread[:, 1]).all() and (spread[:, 1] < 0.08).all()     # about 1 / sqrt(512) = 0.0442
    assert (collapsed[:, :4] < 1e-3).all()


# ------------------------------------------------------------------------------------------ live features
FRAMES = [29, 95, 200, 61, 130, 45]
SIZES = [(171, 128), (160, 121), (171, 128), (173, 131), (171, 128), (149, 113)]


def _trained(k=3):
    m = _model()
    x1, x2, labels = _batch(8, 16, 112, seed=5)
    for _ in range(k):
        m.train_step(x1, x2, labels, LW, lr=0.03)
    return m


def _from_checkpoint(m):
    from cstp_b200 import train
    from cstp_b200.models.model import neq_load_customized
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    path = os.path.join(tempfile.mkdtemp(), "save_3.pth")
    train.save_checkpoint(path, m, 2, "r21d_byol")
    sd = torch.load(path, map_location="cpu", weights_only=False)["state_dict"]
    ft = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
    neq_load_customized(ft, {k[len("module."):]: v for k, v in sd.items()}, verbose=False)
    return ft.cuda().eval()


@pytest.mark.skipif(not features.check_feature("libjpeg_turbo"), reason="the decode contract is Pillow on libjpeg-turbo")
def test_live_features_equal_the_checkpoint_round_trip():
    from cstp_b200.evaluate import video_features, video_features_jpeg
    from tests.test_gpu_finetune_batches import _dataset
    store, read_frames, _ = _dataset(FRAMES, SIZES)
    m = _trained()
    eng = m._engine
    before = _state(m)
    graph = eng._graph
    live = video_features(m, store, FRAMES, capacity=7)
    live_jpeg = video_features_jpeg(m, read_frames, FRAMES, capacity=7)
    after = _state(m)
    assert all(torch.equal(before[k], after[k]) for k in before)       # no running statistic, no counter, no weight
    assert m._engine is eng and eng._graph is graph                      # the captured step is untouched
    ft = _from_checkpoint(m)
    ref = video_features(ft, store, FRAMES, capacity=7)
    assert torch.equal(live, ref) and torch.equal(live_jpeg, ref)
    assert (live.norm(dim=1) > 0).all()
    # one more fused step: the feature engine re-packs the new weights
    x1, x2, labels = _batch(8, 16, 112, seed=6)
    m.train_step(x1, x2, labels, LW, lr=0.03)
    moved = video_features(m, store, FRAMES, capacity=7)
    assert not torch.equal(moved, live)
    assert torch.equal(moved, video_features(_from_checkpoint(m), store, FRAMES, capacity=7))


def test_pretrain_epochs_with_monitor_and_statistics_train_bit_identically():
    from cstp_b200 import train as TR
    from cstp_b200.data_process.datasets import GpuVideoStore
    from tests.test_gpu_video_eval import _synthetic_store
    gallery = _synthetic_store(len(FRAMES))
    query = GpuVideoStore()
    for i, v in enumerate((1, 3, 4)):
        query.put(i, gallery[v])
    opts = types.SimpleNamespace(n_epochs=3, learning_rate=0.03, momentum=0.9, weight_decay=5e-4, clip_grad_norm=1,
                                 loss_weight=list(LW))

    def batches(epoch):
        for s in range(2):
            yield _batch(4, 8, 64, seed=10 * epoch + s)
    mon = TR.RetrievalMonitor((gallery, FRAMES, [0, 1, 2, 3, 4, 5]), (query, [FRAMES[v] for v in (1, 3, 4)], [1, 3, 4]),
                              capacity=16)
    d = tempfile.mkdtemp()
    res = {}
    for on in (False, True):
        path = os.path.join(d, str(on))
        os.makedirs(path)
        m = _model()
        rows = TR.pretrain_epochs(m, batches, opts, result_path=path, collapse_stats=on, monitor=mon if on else None,
                                  monitor_every=1)
        res[on] = (rows, torch.load(os.path.join(path, "save_3.pth"), weights_only=False))
        del m
        torch.cuda.empty_cache()
    (rows_a, ck_a), (rows_b, ck_b) = res[False], res[True]
    for ra, rb in zip(rows_a, rows_b):
        assert [rb[c] for c in TR.LOG_COLUMNS] == [ra[c] for c in TR.LOG_COLUMNS]
        assert all(c in rb for c in ("std_feat", "std_proj", "std_pred", "std_tproj", "feat_norm", "recall@1", "recall@50"))
        assert list(ra) == TR.LOG_COLUMNS
    print(rows_b)
    assert rows_b[-1]["recall@50"] == 1.0                    # the whole gallery holds every query's label
    for k in ck_a["state_dict"]:
        assert torch.equal(ck_a["state_dict"][k], ck_b["state_dict"][k]), k
    for i, st in ck_a["optimizer"]["state"].items():
        assert torch.equal(st["momentum_buffer"], ck_b["optimizer"]["state"][i]["momentum_buffer"])
