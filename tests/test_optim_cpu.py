"""Adam / AdamW on the fused path, without a GPU: the float32 stand-in of the kernel (tests/emulate_adam.py) against
torch.optim.Adam / AdamW, and the engines, drivers and checkpoints over the emulated op layer (tests/emulate_ops.py plus
the stand-in, registered by this file's fixture)."""
import types

import pytest
import torch

from oracle import cstp_oracle as O
from tests import emulate_adam as EA
from tests.parity import rel

LR, BETAS, EPS = 1e-3, (0.9, 0.999), 1e-8


@pytest.fixture()
def emu(monkeypatch):
    from cstp_b200 import engine
    from tests import emulate_ops
    monkeypatch.setattr(engine, "ops", emulate_ops)
    monkeypatch.setattr(engine, "ACT_DTYPE", torch.float32)
    EA.install(monkeypatch)
    return engine


def _close(got, want, tol=1e-6):
    """Per element |got - want| <= tol * (|want| + max |want|).  torch's CPU lerp / addcmul / add(alpha) fuse a
    multiply-add into one rounding where the kernel rounds each operation, so where exp_avg cancels to near zero the two
    differ by an ulp of the terms, not of their sum; the tensor's largest magnitude sets that scale."""
    err = ((got - want).abs() / (want.abs() + want.abs().max())).max().item()
    assert err <= tol, err


@pytest.mark.parametrize("kind", ["adam", "adamw"])
@pytest.mark.parametrize("wd", [0.0, 0.05])
@pytest.mark.parametrize("max_norm", [None, 0.5, 1e6])        # no clipping, clipping active, clipping inactive
def test_standin_matches_torch_adam_over_20_steps(kind, wd, max_norm):
    from cstp_b200.engine import adam_scalars
    g = torch.Generator().manual_seed(7)
    shapes = [(64, 3, 3), (37,), (128,), (1000,)]
    params = [torch.randn(s, generator=g) * 0.05 for s in shapes]
    frozen = 1                                                 # this parameter never gets a gradient: no update, no state
    stream = [[None if i == frozen else torch.randn(s, generator=g) * 0.1 for i, s in enumerate(shapes)] for _ in range(20)]
    rp, rm, rv = EA.torch_reference(params, stream, kind, LR, BETAS, EPS, wd, max_norm)
    assert torch.equal(rp[frozen], params[frozen]) and rm[frozen] is None
    # the fused layout: one flat buffer per tensor kind, the frozen parameter outside the updated ranges
    flat = torch.cat([t.reshape(-1) for t in params])
    m, v = torch.zeros_like(flat), torch.zeros_like(flat)
    offs = [0]
    for t in params:
        offs.append(offs[-1] + t.numel())
    ranges = [(offs[i], offs[i + 1] - offs[i]) for i in range(len(shapes)) if i != frozen]
    for k, grads in enumerate(stream):
        gflat = torch.cat([torch.zeros(s).reshape(-1) if gr is None else gr.reshape(-1) for s, gr in zip(shapes, grads)])
        norm = gflat.double().norm().item()
        coef = EA.clip_coefficient(norm, max_norm or 0.0, max_norm is not None)
        h = adam_scalars(k + 1, LR, BETAS, EPS, wd, kind == "adamw")
        for off, n in ranges:
            EA.adam_update(flat[off:off + n].numpy(), gflat[off:off + n].numpy(), m[off:off + n].numpy(),
                           v[off:off + n].numpy(), coef, h)
    for i in range(len(shapes)):
        sl = slice(offs[i], offs[i + 1])
        if i == frozen:
            assert torch.equal(flat[sl], params[i].reshape(-1)) and not m[sl].any() and not v[sl].any()
            continue
        _close(flat[sl], rp[i].reshape(-1))
        _close(m[sl], rm[i].reshape(-1))
        _close(v[sl], rv[i].reshape(-1))


def test_adam_scalars_are_torchs_double_precision_values():
    from cstp_b200.engine import adam_scalars
    h = adam_scalars(3, 2e-3, (0.8, 0.99), 1e-7, 0.1, False, 18.0, True)
    assert h == (2e-3 / (1 - 0.8 ** 3), (1 - 0.99 ** 3) ** 0.5, 1 - 0.8, 0.99, 1 - 0.99, 1e-7, 0.1, 1.0, 18.0, 1.0)
    hw = adam_scalars(3, 2e-3, (0.8, 0.99), 1e-7, 0.1, True)
    assert hw[6] == 0.0 and hw[7] == 1 - 2e-3 * 0.1 and hw[9] == 0.0


def _pretrain_model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    return R21DBYOL(pretrain=True)


def _torch_group_keys(cls):
    p = torch.nn.Parameter(torch.zeros(2))
    opt = cls([p], lr=LR)
    torch.optim.lr_scheduler.LambdaLR(opt, lambda e: 1.0)      # a scheduler adds initial_lr, as the reference's does
    p.grad = torch.ones(2)
    opt.step()
    sd = opt.state_dict()
    return set(sd["param_groups"][0]), set(sd["state"][0])


@pytest.mark.parametrize("kind", ["adam", "adamw"])
def test_state_dict_loads_into_torch_and_round_trips(emu, kind):
    from cstp_b200 import train as TR
    cls = torch.optim.AdamW if kind == "adamw" else torch.optim.Adam
    m = _pretrain_model()
    x1, x2, lab = O.structured_batch(2, 0, 4, 32)
    for _ in range(2):
        m.train_step(x1, x2, lab, (0.1, 1, 1, 1, 1), lr=LR, optimizer=kind, weight_decay=0.01)
    eng = m._engine
    assert eng.adam_step == 2 and eng.optim_kind == kind
    sd = TR.optimizer_state_dict(m, lr=LR, weight_decay=0.01, initial_lr=3e-3)
    group_keys, state_keys = _torch_group_keys(cls)
    assert set(sd["param_groups"][0]) == group_keys
    names = [n for n, _ in m.named_parameters()]
    assert sorted(sd["state"]) == [i for i, n in enumerate(names) if not n.startswith("target_net.")]
    assert all(set(st) == state_keys and st["step"].item() == 2.0 for st in sd["state"].values())
    probe = _pretrain_model()
    opt = cls(probe.parameters(), lr=LR, weight_decay=0.01)
    opt.load_state_dict(sd)
    g = opt.param_groups[0]
    assert (g["lr"], g["betas"], g["eps"], g["weight_decay"], g["initial_lr"]) == (LR, BETAS, EPS, 0.01, 3e-3)
    i = names.index("predictor.net.0.weight")
    p = list(probe.parameters())[i]
    assert torch.equal(opt.state[p]["exp_avg"], eng.train.view(names[i], eng.exp_avg))
    # one torch step on the loaded state, then back into a fresh engine: moments and step count come along
    for q in probe.parameters():
        if q.requires_grad:
            q.grad = torch.full_like(q, 1e-3)
    opt.step()
    m2 = _pretrain_model()
    m2._bind(x1)
    TR.load_optimizer_state_dict(m2, opt.state_dict())
    e2 = m2._engine
    assert e2.optim_kind == kind and e2.adam_step == 3 and not e2.first_step
    for j in (i, names.index("online_net.conv1.spatial_conv.weight")):
        assert torch.equal(e2.train.view(names[j], e2.exp_avg), opt.state[list(probe.parameters())[j]]["exp_avg"])
        assert torch.equal(e2.train.view(names[j], e2.exp_avg_sq), opt.state[list(probe.parameters())[j]]["exp_avg_sq"])
    # an AdamW file loaded as Adam is the caller's choice; an SGD kind cannot take Adam state
    with pytest.raises(ValueError):
        TR.load_optimizer_state_dict(m2, opt.state_dict(), optimizer="sgd")


def test_sgd_state_dict_is_unchanged_by_default(emu):
    from cstp_b200 import train as TR
    m = _pretrain_model()
    x1, x2, lab = O.structured_batch(2, 0, 4, 32)
    m.train_step(x1, x2, lab, (0.1, 1, 1, 1, 1), lr=0.02)
    sd = TR.optimizer_state_dict(m)
    assert all(set(st) == {"momentum_buffer"} for st in sd["state"].values())
    assert m._engine.exp_avg is None                       # an SGD run allocates no Adam moments


def test_switching_optimizer_kind_raises(emu):
    m = _pretrain_model()
    x1, x2, lab = O.structured_batch(2, 0, 4, 32)
    with pytest.raises(ValueError):
        m.train_step(x1, x2, lab, optimizer="lamb")
    m.train_step(x1, x2, lab, lr=LR, optimizer="adam")
    before = m._engine.train.data.clone()
    for other in ("sgd", "adamw"):
        with pytest.raises(ValueError):
            m.train_step(x1, x2, lab, lr=LR, optimizer=other)
    assert torch.equal(m._engine.train.data, before)          # the refused step changed nothing
    s = _pretrain_model()
    s.train_step(x1, x2, lab, lr=0.02)
    with pytest.raises(ValueError):
        s.train_step(x1, x2, lab, lr=LR, optimizer="adam")


def _opts(n_epochs):
    return types.SimpleNamespace(n_epochs=n_epochs, learning_rate=LR, momentum=0.9, weight_decay=5e-4, clip_grad_norm=1,
                                 loss_weight=[0.1, 1.0, 1.0, 1.0, 1.0])


def test_pretrain_epochs_with_adam_resume_from_checkpoint(emu, tmp_path):
    from cstp_b200 import train as TR

    def batches(epoch):
        for s in range(2):
            yield O.structured_batch(2, 10 * epoch + s, 4, 32)

    a = _pretrain_model()
    rows_a = TR.pretrain_epochs(a, batches, _opts(3), result_path=str(tmp_path), save_every=2, optimizer="adamw",
                                betas=(0.85, 0.995))
    assert [r["epoch"] for r in rows_a] == [1, 2, 3] and a._engine.adam_step == 6
    ck = torch.load(tmp_path / "save_2.pth", weights_only=False)
    g = ck["optimizer"]["param_groups"][0]
    assert g["betas"] == (0.85, 0.995) and g["decoupled_weight_decay"] is True
    assert all(st["step"].item() == 4.0 for st in ck["optimizer"]["state"].values())
    b = _pretrain_model()
    x1 = O.structured_batch(2, 0, 4, 32)[0]
    begin = TR.load_checkpoint(str(tmp_path / "save_2.pth"), b, example_clip=x1)
    assert begin == 2 and b._engine.optim_kind == "adamw" and b._engine.adam_step == 4
    rows_b = TR.pretrain_epochs(b, batches, _opts(3), begin_epoch=3, optimizer="adamw", betas=(0.85, 0.995))
    assert abs(rows_b[0]["loss"] - rows_a[2]["loss"]) <= 1e-6 * abs(rows_a[2]["loss"])
    sa, sb = a.state_dict(), b.state_dict()
    assert max(rel(sa[k], sb[k]) for k in sa if sa[k].dtype.is_floating_point) < 1e-6


def _ft_model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    return R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)


@pytest.mark.parametrize("kind", ["adam", "adamw"])
def test_fused_finetune_step_matches_torch_adam_with_frozen_backbone(emu, kind):
    from cstp_b200.models.pace.r21d_byol import get_fine_tuning_parameters
    cls = torch.optim.AdamW if kind == "adamw" else torch.optim.Adam
    x = O.structured_batch(2, 1, 4, 32)[0]
    labels = torch.tensor([3, 77])
    for freeze in (False, True):
        a, b = _ft_model(), _ft_model()
        a.train()
        b.train()
        if freeze:
            get_fine_tuning_parameters(a, 5)
        groups = get_fine_tuning_parameters(b, 5) if freeze else b.parameters()
        before = {n: p.detach().clone() for n, p in a.named_parameters()}
        # one step from the same weights: the same gradients, so only the two optimisers' rounding differs (Adam's
        # first steps amplify later gradient differences in elements whose gradient is near zero)
        a.finetune_step(x, labels, lr=LR, weight_decay=1e-2, optimizer=kind)
        opt = cls(groups, lr=LR, weight_decay=1e-2, foreach=False)
        lb = torch.nn.CrossEntropyLoss()(b(x, o_type="ft_fc" if freeze else "ft_all"), labels)
        opt.zero_grad()
        lb.backward()
        opt.step()
        sa, sb = a.state_dict(), b.state_dict()
        assert max(rel(sa[k], sb[k]) for k in sa if sa[k].dtype.is_floating_point) < 1e-5
        from cstp_b200 import train as TR
        sd = TR.optimizer_state_dict(a, lr=LR, weight_decay=1e-2)
        assert len(sd["state"]) == len(opt.state)                  # frozen parameters: no state, as torch gives them none
        a.finetune_step(x, labels, lr=LR, weight_decay=1e-2, optimizer=kind)
        for n, p in a.named_parameters():
            if freeze and not n.startswith("classify."):
                assert torch.equal(p, before[n]), n                # no update, no weight decay
                assert not a._engine.train.view(n, a._engine.exp_avg).any()
            elif n.startswith("classify."):
                assert not torch.equal(p, before[n]), n


def test_finetune_epochs_with_adam_keep_the_best_checkpoint(emu, tmp_path):
    from cstp_b200 import train as TR
    data = [(O.structured_batch(2, s, 4, 32)[0], torch.tensor([3 + s, 77 - s])) for s in range(2)]
    m = _ft_model()
    opts = types.SimpleNamespace(n_epochs=2, learning_rate=LR, momentum=0.9, weight_decay=1e-3, lr_patience=0,
                                 task="ft_all", highest_val={"name": -1.0})
    rows_t, rows_v = TR.finetune_epochs(m, lambda e: iter(data), lambda e: iter(data[:1]), opts,
                                        result_path=str(tmp_path), optimizer="adam")
    assert [r["epoch"] for r in rows_t] == [1, 2] and m._engine.adam_step == 4
    files = [p.name for p in tmp_path.iterdir()]
    assert len(files) == 1
    ck = torch.load(tmp_path / files[0], weights_only=False)
    assert all(set(st) == {"step", "exp_avg", "exp_avg_sq"} for st in ck["optimizer"]["state"].values())
