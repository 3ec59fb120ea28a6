"""The standalone R2Plus1DNet (models.pace.r21d_byol) on CPU: its engine (cstp_b200.engine_backbone) runs on the torch
restatement of the op layer (tests/emulate_backbone.py, fp32 storage) and is compared with the oracle's r2plus1d_net
under torch autograd; the stem input-gradient stand-in is checked against torch.nn.grad.conv3d_input in float64."""
import os

import pytest
import torch
import torch.nn.functional as F

from oracle import cstp_oracle as O
from tests.emulate_backbone import stem_dgrad_reference
from tests.parity import rel

B, T, S = 2, 4, 32


@pytest.fixture()
def emu():
    from cstp_b200 import engine
    from tests import emulate_backbone
    saved = engine.ops, engine.ACT_DTYPE
    engine.ops, engine.ACT_DTYPE = emulate_backbone, torch.float32
    torch.set_num_threads(os.cpu_count() or 1)
    try:
        yield engine
    finally:
        engine.ops, engine.ACT_DTYPE = saved


def _net(proj=False, seed=0):
    from cstp_b200.models.pace.r21d_byol import R2Plus1DNet
    torch.manual_seed(seed)
    net = R2Plus1DNet((1, 1, 1, 1), proj_flag=proj)
    with torch.no_grad():                    # non-trivial BatchNorm affine maps and running statistics
        for name, b in net.named_buffers():
            if name.endswith("running_mean"):
                b.uniform_(-0.1, 0.1)
            elif name.endswith("running_var"):
                b.uniform_(0.5, 1.5)
        for name, p in net.named_parameters():
            if p.dim() == 1 and ".bias" in name:
                p.uniform_(-0.1, 0.1)
    return net


def _clips(n=B, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(n, 3, T, S, S, generator=g)


def _state(net):
    return {k: v.detach().clone() for k, v in net.state_dict().items() if not k.endswith("num_batches_tracked")}


def _oracle(state, xs, proj, need_x_grad=False):
    """r2plus1d_net on each clip batch in order (BatchNorm buffers carried over); returns outputs, parameter / input
    gradients of sum(out * upstream) and the final buffers."""
    params = {k: v.clone().requires_grad_("running" not in k) for k, v in state.items()}
    bufs: dict = {}
    P = O._ParamView({"net." + k: v for k, v in params.items()}, bufs)
    xs = [x.clone().requires_grad_(need_x_grad) for x in xs]
    outs = [O.r2plus1d_net(x, P, "net", bufs, O.Tape(False), f"v{i}", proj=proj) for i, x in enumerate(xs)]
    return params, xs, outs, {k[len("net."):]: v for k, v in bufs.items()}


def _upstreams(n_calls, proj, seed=5):
    g = torch.Generator().manual_seed(seed)
    return [(torch.randn(B, 512, generator=g), torch.randn(B, 512, generator=g) if proj else None) for _ in range(n_calls)]


def _loss(outs, ups, proj):
    tot = 0
    for o, (uf, up) in zip(outs, ups):
        if proj:
            tot = tot + (o[0] * uf).sum() + (o[1] * up).sum()
        else:
            tot = tot + (o * uf).sum()
    return tot


def _grad_errors(net, params):
    # (a Linear bias in front of a BatchNorm has a zero gradient up to rounding: skip gradients that small)
    total = sum(params[n].grad.double().pow(2).sum() for n, _ in net.named_parameters()).sqrt().item()
    errs = {n: rel(p.grad, params[n].grad) for n, p in net.named_parameters() if params[n].grad.norm() > 1e-4 * total}
    return sorted(errs.values())[len(errs) // 2], max(errs.values()), errs


@pytest.mark.parametrize("proj", [False, True])
def test_train_call_matches_oracle(emu, proj):
    net = _net(proj)
    state = _state(net)
    x = _clips()
    xg = x.clone().requires_grad_(True)
    out = net(xg)
    ups = _upstreams(1, proj)
    _loss([out], ups, proj).backward()
    params, xs, ref, bufs = _oracle(state, [x], proj, need_x_grad=True)
    _loss(ref, ups, proj).backward()
    if proj:
        assert rel(out[0], ref[0][0]) < 1e-4 and rel(out[1], ref[0][1]) < 1e-4
    else:
        assert rel(out, ref[0]) < 1e-4
    med, worst, errs = _grad_errors(net, params)
    assert med < 1e-2 and worst < 5e-2, sorted(errs.items(), key=lambda kv: -kv[1])[:4]
    # the stem input gradient rounds the weight to bf16 (as the packed weights of every dgrad are)
    assert xg.grad is not None and xg.grad.shape == x.shape
    assert rel(xg.grad, xs[0].grad) < 1e-2
    sd = net.state_dict()
    for k, v in bufs.items():
        assert rel(sd[k], v) < 1e-4, k
    assert all(v.item() == 1 for k, v in sd.items() if k.endswith("num_batches_tracked"))
    assert len(net._pools[(B, T, S, S, torch.device("cpu"), "grad")]) == 1       # the arena is back in its pool


def test_two_calls_one_backward_sum_gradients_and_update_statistics_in_order(emu):
    net = _net(True)
    state = _state(net)
    x1, x2 = _clips(seed=1), _clips(seed=2)
    o1, o2 = net(x1), net(x2)
    assert len(net._pools[(B, T, S, S, torch.device("cpu"), "grad")]) == 0        # two live arenas
    ups = _upstreams(2, True)
    _loss([o1, o2], ups, True).backward()
    params, _, ref, bufs = _oracle(state, [x1, x2], True)
    _loss(ref, ups, True).backward()
    assert rel(o1[0], ref[0][0]) < 1e-4 and rel(o2[1], ref[1][1]) < 1e-4
    med, worst, errs = _grad_errors(net, params)
    assert med < 1e-2 and worst < 5e-2, sorted(errs.items(), key=lambda kv: -kv[1])[:4]
    sd = net.state_dict()
    for k, v in bufs.items():
        assert rel(sd[k], v) < 1e-4, k
    assert sd["bn1.num_batches_tracked"].item() == 2 and sd["project.net.1.num_batches_tracked"].item() == 2
    assert len(net._pools[(B, T, S, S, torch.device("cpu"), "grad")]) == 2


def test_no_grad_call_updates_statistics_and_keeps_no_arena(emu):
    net = _net(False)
    state = _state(net)
    x = _clips()
    with torch.no_grad():
        out = net(x)
    assert out.grad_fn is None
    _, _, ref, bufs = _oracle(state, [x], False)
    assert rel(out, ref[0]) < 1e-4
    sd = net.state_dict()
    for k, v in bufs.items():
        assert rel(sd[k], v) < 1e-4, k
    assert sd["conv5.block1.bn2.num_batches_tracked"].item() == 1
    assert list(net._pools) == [(B, T, S, S, torch.device("cpu"), "nograd")]
    assert len(net._pools[(B, T, S, S, torch.device("cpu"), "nograd")]) == 1


def test_dropped_output_returns_its_arena(emu):
    net = _net(False)
    key = (B, T, S, S, torch.device("cpu"), "grad")
    out = net(_clips())
    assert len(net._pools[key]) == 0
    del out
    assert len(net._pools[key]) == 1
    out = net(_clips())                      # the pooled arena is reused
    out.sum().backward()
    assert len(net._pools[key]) == 1


@pytest.mark.parametrize("proj", [False, True])
def test_eval_features_use_running_statistics(emu, proj, monkeypatch):
    net = _net(proj)
    state = _state(net)
    net.eval()
    x = _clips(3)
    with torch.no_grad():
        out = net(x)

    def bn_eval(x, P, name, buffers_out, tape, tag):
        return F.batch_norm(x, P[name + ".running_mean"], P[name + ".running_var"], P[name + ".weight"],
                            P[name + ".bias"], False, 0.1, 1e-5)
    monkeypatch.setattr(O, "_bn", bn_eval)
    with torch.no_grad():
        P = {"net." + k: v for k, v in state.items()}
        ref = O.r2plus1d_net(x, P, "net", {}, O.Tape(False), "e", proj=proj)
    if proj:
        assert out[0].shape == (3, 512) and rel(out[0], ref[0]) < 1e-4 and rel(out[1], ref[1]) < 1e-4
    else:
        assert out.shape == (3, 512) and rel(out, ref) < 1e-4
    sd = net.state_dict()
    assert all(v.item() == 0 for k, v in sd.items() if k.endswith("num_batches_tracked"))
    assert all(torch.equal(sd[k], v) for k, v in state.items())
    assert (4, T, S, S, torch.device("cpu"), "eval") in net._pools       # capacity bucket of 3 clips


def test_optimizer_step_and_load_state_dict_reach_the_next_call(emu):
    net = _net(False)
    x = _clips()
    opt = torch.optim.SGD(net.parameters(), lr=0.1)
    net(x).sum().backward()
    opt.step()
    with torch.no_grad():
        a = net(x)
        fresh = _net(False, seed=3)
        fresh.load_state_dict(net.state_dict())
        b = fresh(x)
    assert torch.equal(a, b)
    with torch.no_grad():
        net.load_state_dict(_net(False, seed=7).state_dict())
        c = net(x)
    assert not torch.equal(a, c)


def _fresh_like(net, proj, grad, x):
    """The same call on a new module loaded with net's current state_dict (its engines are built and packed anew)."""
    fresh = _net(proj, seed=3)
    fresh.load_state_dict({k: v.clone() for k, v in net.state_dict().items()})
    if grad:
        return fresh(x)
    with torch.no_grad():
        return fresh(x)


def _pool_len(net, variant):
    return len(net._pools.get((B, T, S, S, torch.device("cpu"), variant), []))


def test_sgd_step_reaches_the_next_grad_call_on_the_pooled_engine(emu):
    net = _net(True)
    x = _clips()
    opt = torch.optim.SGD(net.parameters(), lr=0.1, momentum=0.9)
    for _ in range(2):
        f, p = net(x)
        (f.square().mean() + p.square().mean()).backward()
        opt.step()
        opt.zero_grad()
    assert _pool_len(net, "grad") == 1           # the next grad call reuses the engine packed before the step
    want = _fresh_like(net, True, True, x)
    got = net(x)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_in_place_target_update_reaches_the_next_no_grad_call(emu):
    online, target = _net(True), _net(True, seed=4)
    x = _clips()
    with torch.no_grad():
        target(x)
    assert _pool_len(target, "nograd") == 1
    with torch.no_grad():                        # the BYOL target update (r21d_byol.py:331-337), in place
        for pt, po in zip(target.parameters(), online.parameters()):
            pt.mul_(0.5).add_(po, alpha=0.5)
    want = _fresh_like(target, True, False, x)
    with torch.no_grad():
        got = target(x)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_data_assignment_and_marked_data_writes_reach_the_next_call(emu):
    net = _net(False)
    x = _clips()
    with torch.no_grad():
        net(x)
        w = net.conv3.block1.conv1.spatial_conv.weight
        w.data = w.data * 0.5                    # re-assignment: the parameter leaves the engine's store
        want = _fresh_like(net, False, False, x)
        got = net(x)
    assert torch.equal(got, want)
    with torch.no_grad():
        net.conv4.block1.conv2.temporal_conv.weight.data.mul_(2.0)     # behind autograd's back: announced
        net.mark_weights_dirty()
        want = _fresh_like(net, False, False, x)
        got = net(x)
    assert torch.equal(got, want)


def test_state_dict_keys_are_the_references():
    from cstp_b200.engine import backbone_param_specs
    from cstp_b200.models.pace.r21d_byol import R2Plus1DNet
    for proj in (False, True):
        net = R2Plus1DNet((1, 1, 1, 1), proj_flag=proj)
        specs = backbone_param_specs("x", project=proj)
        assert [(n, tuple(p.shape)) for n, p in net.named_parameters()] == [(n[2:], s) for n, s in specs]
        keys = list(net.state_dict())
        assert all(k.endswith(("weight", "bias", "running_mean", "running_var", "num_batches_tracked")) for k in keys)
        assert ("project.net.3.weight" in keys) == proj and "conv1.bn.running_var" in keys


def test_errors(emu):
    from cstp_b200.models.pace.r21d_byol import (R21DBYOL, Predictor, Projector, R2Plus1DNet, SpatioTemporalConv,
                                                 SpatioTemporalResBlock)
    m = R21DBYOL(pretrain=True)
    for sub in (m.online_net, m.target_net):
        with pytest.raises(RuntimeError, match="video_features"):
            sub(_clips())
    with pytest.raises(RuntimeError, match="video_features"):
        R21DBYOL(pretrain=False, num_classes=5, cls_bn=True).online_net(_clips())
    for holder in (SpatioTemporalConv(3, 8, 3), SpatioTemporalResBlock(8, 8, 3), Projector(8, 8, 8), Predictor(8, 8, 8)):
        with pytest.raises(RuntimeError, match="only holds parameters"):
            holder(torch.zeros(1))
    with pytest.raises(ValueError):
        R2Plus1DNet((2, 2, 2, 2))
    net = _net(False)
    with pytest.raises(Exception, match="multiple of 4"):
        net(torch.zeros(B, 3, T, S, S - 2))
    net.eval()
    with pytest.raises(Exception, match="forward only"):
        net(_clips().requires_grad_(True))


def test_cpu_tensors_raise_cstp_error():
    from cstp_b200.lib import CstpError
    net = _net(False)
    with pytest.raises(CstpError):
        net(_clips())


@pytest.mark.parametrize("H,W,cout,Cg", [(32, 32, 83, 96), (14, 20, 5, 16), (8, 68, 84, 96)])
def test_stem_input_gradient_stand_in_matches_conv3d_input(H, W, cout, Cg):
    g = torch.Generator().manual_seed(H * W + cout)
    N, Tn = 2, 3
    d = torch.randn(N, Tn, H // 2, W // 2, Cg, generator=g).to(torch.bfloat16)
    d[..., cout:] = 0
    w = torch.randn(cout, 3, 1, 7, 7, generator=g) * 0.1
    got = stem_dgrad_reference(d, w, H, W)
    wb = w.to(torch.bfloat16).double()
    gd = d[..., :cout].double().permute(0, 4, 1, 2, 3)
    ref = torch.nn.grad.conv3d_input((N, 3, Tn, H, W), wb, gd, stride=(1, 2, 2), padding=(0, 3, 3))
    assert got.shape == ref.shape
    assert ((got.double() - ref).abs().max() / ref.abs().max()).item() < 1e-6
