"""Adam / AdamW on the GPU: cstp_adam_clip_step against its float32 stand-in (tests/emulate_adam.py) bit for bit at the
size of the pretraining buffers, against torch.optim.Adam / AdamW on the same device, and through the fused pretraining
and finetune steps, the captured graph and the checkpoints."""
import numpy as np
import pytest
import torch

from tests import emulate_adam as EA
from tests.parity import rel
from tests.test_optim_cpu import BETAS, EPS, _close

pytestmark = pytest.mark.gpu

LW = (0.1, 1.0, 1.0, 1.0, 1.0)


def _pretrain_numel():
    from cstp_b200.engine import FlatStore, trainable_param_specs
    return FlatStore(trainable_param_specs(), "meta").numel


def _buffers(n, seed):
    r = np.random.default_rng(seed)
    p = (r.standard_normal(n, dtype=np.float32) * np.float32(0.05))
    m = (r.standard_normal(n, dtype=np.float32) * np.float32(1e-3))
    v = (r.random(n, dtype=np.float32) * np.float32(1e-5))
    return p, m, v


def _run_kernel(kind, n, steps, wd, max_norm, dev=False, seed=0):
    """`steps` steps of the kernel from seeded buffers; returns (p, m, v, [(norm, coef) per step]) and the stand-in's
    (p, m, v) from the same start, each step applied with the kernel's clip coefficient."""
    from cstp_b200 import ops
    from cstp_b200.engine import adam_scalars
    p, m, v = _buffers(n, seed)
    dp, dm, dv = (torch.from_numpy(a).cuda() for a in (p, m, v))
    norm_out, ws = torch.zeros(2, device="cuda"), torch.zeros(2048, device="cuda")
    hyper = torch.zeros(ops.ADAM_HYPER_FLOATS, device="cuda")
    r = np.random.default_rng(seed + 1)
    norms = []
    for t in range(1, steps + 1):
        g = r.standard_normal(n, dtype=np.float32) * np.float32(1e-3)
        h = adam_scalars(t + 10, 1e-3, BETAS, EPS, wd, kind == "adamw", max_norm or 0.0, max_norm is not None)
        dg = torch.from_numpy(g).cuda()
        if dev:
            hyper.copy_(torch.tensor(h, dtype=torch.float32))
            ops.adam_clip_step_dev(dp, dg, dm, dv, hyper, norm_out, ws)
        else:
            ops.adam_clip_step(dp, dg, dm, dv, h, norm_out, ws)
        norm, coef = norm_out.tolist()
        norms.append((norm, coef, float(np.linalg.norm(g.astype(np.float64)))))
        EA.adam_update(p, g, m, v, np.float32(coef), h)
    return (dp.cpu().numpy(), dm.cpu().numpy(), dv.cpu().numpy()), (p, m, v), norms


@pytest.mark.parametrize("kind", ["adam", "adamw"])
def test_kernel_equals_standin_bit_for_bit_on_pretraining_size(kind):
    n = _pretrain_numel()
    assert 25_400_000 < n < 25_500_000
    for size, dev in ((n, False), (n - 3, True)):                  # n - 3: the n % 4 tail, and the device-scalar form
        got, want, norms = _run_kernel(kind, size, 3, 0.05, 0.02, dev=dev)
        for a, b in zip(got, want):
            assert np.array_equal(a.view(np.uint32), b.view(np.uint32))
        for norm, coef, ref in norms:
            assert abs(norm - ref) <= 1e-5 * ref
            assert coef == EA.clip_coefficient(norm, 0.02, True) and coef < 1.0        # clipping active
    again, _, _ = _run_kernel(kind, n, 3, 0.05, 0.02)
    got, _, _ = _run_kernel(kind, n, 3, 0.05, 0.02)
    for a, b in zip(got, again):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))          # run to run: identical bits


@pytest.mark.parametrize("kind", ["adam", "adamw"])
@pytest.mark.parametrize("wd,max_norm", [(0.0, None), (0.05, 0.5), (0.05, 1e6)])
def test_kernel_tracks_torch_adam_on_the_device(kind, wd, max_norm):
    from cstp_b200 import ops
    from cstp_b200.engine import adam_scalars
    g = torch.Generator().manual_seed(3)
    shapes = [(256, 64, 3), (300,), (4096,)]
    params = [torch.randn(s, generator=g) * 0.05 for s in shapes]
    stream = [[torch.randn(s, generator=g) * 0.1 for s in shapes] for _ in range(20)]
    rp, rm, rv = EA.torch_reference(params, stream, kind, 1e-3, BETAS, EPS, wd, max_norm, device="cuda")
    offs = np.cumsum([0] + [t.numel() for t in params])
    pad = lambda k: (k + 3) // 4 * 4
    slots = [pad(k) for k in np.diff(offs)]
    starts = np.cumsum([0] + slots)
    flat = torch.zeros(int(starts[-1]), device="cuda")
    for s0, t in zip(starts, params):
        flat[s0:s0 + t.numel()] = t.reshape(-1).cuda()
    m, v, gf = torch.zeros_like(flat), torch.zeros_like(flat), torch.zeros_like(flat)
    norm_out, ws = torch.zeros(2, device="cuda"), torch.zeros(2048, device="cuda")
    for k, grads in enumerate(stream):
        for s0, gr in zip(starts, grads):
            gf[s0:s0 + gr.numel()] = gr.reshape(-1).cuda()
        h = adam_scalars(k + 1, 1e-3, BETAS, EPS, wd, kind == "adamw", max_norm or 0.0, max_norm is not None)
        ops.adam_clip_step(flat, gf, m, v, h, norm_out, ws)
    for s0, a, b, c in zip(starts, rp, rm, rv):
        sl = slice(int(s0), int(s0) + a.numel())
        _close(flat[sl].cpu(), a.reshape(-1))
        _close(m[sl].cpu(), b.reshape(-1))
        _close(v[sl].cpu(), c.reshape(-1))


def test_wrappers_reject_bad_buffers():
    from cstp_b200 import ops
    from cstp_b200.lib import CstpError
    n = 64
    p, g, m, v = (torch.zeros(n, device="cuda") for _ in range(4))
    no, ws = torch.zeros(2, device="cuda"), torch.zeros(2048, device="cuda")
    h = (1e-3, 1.0, 0.1, 0.999, 0.001, 1e-8, 0.0, 1.0, 0.0, 0.0)
    for bad in ((p.cpu(), g, m, v), (p, g.double(), m, v), (p, g, m[:-4], v), (p, g, m, v[1:].clone()[:0])):
        with pytest.raises(CstpError):
            ops.adam_clip_step(*bad, h, no, ws)
    with pytest.raises(CstpError):
        ops.adam_clip_step(p[1:], g[1:], m[1:], v[1:], h, no, ws)         # not 16-byte aligned
    with pytest.raises(CstpError):
        ops.adam_clip_step_dev(p, g, m, v, torch.zeros(4, device="cuda"), no, ws)


def _model(options=None):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=True)
    m.engine_options = dict(options or {})
    return m.cuda()


def _batch(B, seed):
    from oracle import cstp_oracle as O
    x1, x2, lab = O.structured_batch(B, seed, 8, 64)
    return x1.cuda(), x2.cuda(), tuple(t.cuda() for t in lab)


def test_graphed_adam_step_is_bit_identical_to_eager_launches():
    batches = [_batch(3, s) for s in (5, 6)]
    outs = []
    for graph in (False, True):
        m = _model({"graph": graph})
        losses = []
        for i in range(5):
            l = m.train_step(*batches[i % 2], LW, lr=1e-3 if i < 3 else 3e-4, weight_decay=0.05, optimizer="adam")
            losses.append(l.clone())
        eng = m._engine
        assert (eng._graph is not None) == graph and eng.adam_step == 5
        outs.append((torch.stack(losses), eng.train.data.clone(), eng.target.data.clone(), eng.bufs.data.clone(),
                     eng.exp_avg.clone(), eng.exp_avg_sq.clone(), eng.norm_out.clone()))
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _dropin_step(b, opt, batch):
    crit = torch.nn.CrossEntropyLoss()
    loss_byol, preds = b(batch[0], batch[1], o_type="loss_com")
    spa, tem, pb, r1, r2 = batch[2]
    ce = [crit(preds[0], spa), crit(preds[1], tem), crit(preds[2], pb), crit(preds[3], pb), crit(preds[4], r1), crit(preds[5], r2)]
    total = LW[0] * loss_byol + LW[1] * ce[0] + LW[2] * ce[1] + LW[3] * (ce[2] + ce[3]) + LW[4] * (ce[4] + ce[5])
    opt.zero_grad()
    total.backward()
    gn = torch.nn.utils.clip_grad_norm_(b.parameters(), 18)
    opt.step()
    return loss_byol, gn


def test_fused_adamw_step_equals_dropin_autograd_loop():
    batch = _batch(2, 3)
    a, b = _model({"fuse_min_positions": 0}), _model({"fuse_min_positions": 0})
    la = a.train_step(*batch, LW, lr=1e-3, weight_decay=0.05, optimizer="adamw").clone()
    opt = torch.optim.AdamW(b.parameters(), lr=1e-3, weight_decay=0.05, foreach=False)
    loss_byol, gn = _dropin_step(b, opt, batch)
    assert abs(loss_byol.item() - la[7].item()) < 1e-6
    assert abs(gn.item() - a._engine.norm_out[0].item()) / gn.item() < 1e-4
    sa, sb = a.state_dict(), b.state_dict()
    worst = max(rel(sa[k], sb[k]) for k in sa if sa[k].dtype.is_floating_point)
    assert worst < 1e-5, worst


def test_finetune_adam_ft_fc_updates_only_classify():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL, get_fine_tuning_parameters
    from oracle import cstp_oracle as O
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda()
    m.train()
    get_fine_tuning_parameters(m, 5)
    x = O.structured_batch(4, 1, 8, 64)[0].cuda()
    labels = torch.tensor([3, 77, 5, 100], device="cuda")
    before = {n: p.detach().clone() for n, p in m.named_parameters()}
    for _ in range(3):
        m.finetune_step(x, labels, lr=1e-3, weight_decay=1e-3, optimizer="adam")
    eng = m._engine
    for n, p in m.named_parameters():
        if n.startswith("classify."):
            assert not torch.equal(p, before[n]), n
        else:
            assert torch.equal(p, before[n]), n
            assert not eng.train.view(n, eng.exp_avg).any() and not eng.train.view(n, eng.exp_avg_sq).any()
    from cstp_b200 import train as TR
    assert sorted(TR.optimizer_state_dict(m, lr=1e-3)["state"]) == [i for i, (n, _) in enumerate(m.named_parameters())
                                                                      if n.startswith("classify.")]


def test_checkpoint_interop_with_torch_adam_both_ways(tmp_path):
    from cstp_b200 import train as TR
    batches = [_batch(2, s) for s in (7, 8, 9)]
    kw = dict(lr=1e-3, weight_decay=0.05)
    # fused for two steps -> checkpoint -> reference-style module + torch.optim.Adam takes the third step
    a = _model()
    for bt in batches[:2]:
        a.train_step(*bt, LW, optimizer="adam", **kw)
    TR.save_checkpoint(str(tmp_path / "save_2.pth"), a, 2, "r21d_byol-1", lr=1e-3, weight_decay=0.05)
    ck = torch.load(tmp_path / "save_2.pth", weights_only=False)
    b = _model()
    b.load_state_dict({k[len("module."):]: v for k, v in ck["state_dict"].items()})
    opt = torch.optim.Adam(b.parameters(), lr=1e-3, weight_decay=0.05, foreach=False)
    opt.load_state_dict(ck["optimizer"])
    _dropin_step(b, opt, batches[2])
    a.train_step(*batches[2], LW, optimizer="adam", **kw)
    sa, sb = a.state_dict(), b.state_dict()
    worst = max(rel(sa[k], sb[k]) for k in sa if sa[k].dtype.is_floating_point)
    assert worst < 1e-5, worst
    # and back: torch.optim.Adam state after three drop-in steps -> the fused step continues it
    c = _model()
    c.load_state_dict(b.state_dict())
    c._bind(batches[0][0])
    TR.load_optimizer_state_dict(c, opt.state_dict())
    assert c._engine.adam_step == 3 and c._engine.optim_kind == "adam"
    c.train_step(*batches[0], LW, optimizer="adam", **kw)
    _dropin_step(b, opt, batches[0])
    sc, sb = c.state_dict(), b.state_dict()
    worst = max(rel(sc[k], sb[k]) for k in sc if sc[k].dtype.is_floating_point)
    assert worst < 1e-5, worst


def test_sgd_steps_allocate_no_adam_state_and_launch_as_before():
    from cstp_b200 import ops
    batch = _batch(2, 4)
    m = _model({"graph": False})
    m.train_step(*batch, LW, lr=0.03)
    eng = m._engine
    torch.cuda.synchronize()
    n0 = ops.launch_count()
    eng.optimizer_step(0.03)
    n_sgd = ops.launch_count() - n0
    assert eng.exp_avg is None and eng.exp_avg_sq is None and eng.optim_kind == "sgd"
    a = _model({"graph": False})
    a.train_step(*batch, LW, lr=1e-3, optimizer="adam")
    n0 = ops.launch_count()
    a._engine.optimizer_step(1e-3, optimizer="adam")
    assert ops.launch_count() - n0 == n_sgd                    # norm pass + update + re-pack, for either optimiser
