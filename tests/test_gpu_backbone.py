"""The standalone R2Plus1DNet on the B200 (cstp_b200.engine_backbone): every layer, forward and backward, and the stem
input gradient against fp32 torch operators on the engine's own inputs; eval features bit-identical to FeatureEngine;
train-mode features, running statistics and gradients bit-identical to FinetuneEngine's; a plain-PyTorch BYOL step on
two standalone networks against R21DBYOL.train_step; the input-gradient kernel bit-exact against its float32 stand-in
(tests/emulate_backbone.py); optimiser updates seen by the next call; memory flat over repeated calls."""
import pytest
import torch
import torch.nn.functional as F

from tests import local_parity as LP
from tests.emulate_backbone import stem_dgrad_reference

pytestmark = pytest.mark.gpu
B, T, S = 4, 8, 64


def _net(proj, seed=0):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL, R2Plus1DNet
    torch.manual_seed(seed)
    ref = R21DBYOL(pretrain=True)               # glorot-initialised weights, as a pretraining run starts
    net = R2Plus1DNet((1, 1, 1, 1), proj_flag=proj)
    sd = {k[len("online_net."):]: v for k, v in ref.state_dict().items() if k.startswith("online_net.")}
    if not proj:
        sd = {k: v for k, v in sd.items() if not k.startswith("project.")}
    net.load_state_dict(sd)
    return net.cuda().train()


def _clips(n=B, seed=1, t=T, s=S):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.rand(n, 3, t, s, s, device="cuda", generator=g) * 2 - 1


def _pooled(net, variant, n=B):
    return net._pools[(n, T, S, S, torch.device("cuda", torch.cuda.current_device()), variant)][0]


# ------------------------------------------------------------------------------------------ 1. per layer
def test_every_layer_and_the_input_gradient_against_fp32_torch():
    net = _net(True)
    net.engine_options = {"record": True, "fuse_min_positions": 0}
    params = {"online_net." + k: v.detach().float().cpu().clone() for k, v in net.state_dict().items()}
    x = _clips().requires_grad_(True)
    feat, proj = net(x)
    g = torch.Generator(device="cuda").manual_seed(3)
    (feat * torch.randn(feat.shape, device="cuda", generator=g)).sum().add_(
        (proj * torch.randn(proj.shape, device="cuda", generator=g)).sum()).backward()
    torch.cuda.synchronize()
    eng = _pooled(net, "grad")
    res = LP.check_conv_units(eng, params, "online")
    res["mlp:online.project"] = LP.check_mlp(eng, params, "online.project", "online_net.project.net", 512, 4096, 512, 1)
    # the stem input gradient from the engine's own d(raw)
    g_e = LP._ncdhw(eng.named["online.conv1.spatial.g"], 83)
    ref = torch.nn.grad.conv3d_input(tuple(x.shape), params["online_net.conv1.spatial_conv.weight"], g_e,
                                     stride=(1, 2, 2), padding=(0, 3, 3))
    res["stem:input_grad"] = {"dx": LP.rel(x.grad, ref)}
    assert len([t for t in res if not t.startswith(("dx:", "mlp:", "stem:"))]) == 24
    w = LP.worst(res)
    assert w[0] < 1e-2, w


# ------------------------------------------------------------------------------------------ 2. eval
def test_eval_features_are_bit_identical_to_the_feature_engine():
    from cstp_b200 import engine_ft
    from cstp_b200.models.pace.r21d_byol import R21DBYOL, R2Plus1DNet
    torch.manual_seed(0)
    m = R21DBYOL(pretrain=True).cuda().train()
    x1, x2 = _clips(seed=4), _clips(seed=5)
    labels = tuple(torch.randint(0, 5, (B,), device="cuda") for _ in range(5))
    m.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=0.03)           # non-trivial running statistics
    net = R2Plus1DNet((1, 1, 1, 1))
    net.load_state_dict({k[len("online_net."):]: v for k, v in m.state_dict().items()
                         if k.startswith("online_net.") and ".project." not in k})
    net.cuda().eval()
    for n in (1, 3, 7):
        x = _clips(n, seed=10 + n)
        with torch.no_grad():
            got = net(x)
        cap = engine_ft.inference_capacity(n)
        fe = engine_ft.FeatureEngine(cap, T, S, S, device="cuda", share=m._engine)
        fe.pack_online()
        fe.forward_batch(x)
        assert torch.equal(got, fe.feat[:n]), n


# ------------------------------------------------------------------------------------------ 3. train vs FinetuneEngine
def test_train_call_is_bit_identical_to_the_finetune_engine():
    from cstp_b200.engine_ft import FinetuneEngine
    net = _net(False)
    sd0 = {k: v.clone() for k, v in net.state_dict().items()}
    fe = FinetuneEngine(B, T, S, S, device="cuda", num_classes=5, cls_bn=True)
    for k, v in sd0.items():
        if k.endswith("num_batches_tracked"):
            continue
        (fe.bufs if "running" in k else fe.train).view("online_net." + k).copy_(v)
    fe.pack_online()
    x = _clips(seed=6)
    fe.eval_mode = False
    fe.forward(x)
    fe.cross_entropy(torch.randint(0, 5, (B,), device="cuda"))
    fe.backward()
    feat = net(x)
    feat.backward(fe.dfeat.clone())
    torch.cuda.synchronize()
    assert torch.equal(feat, fe.feat)
    sd = net.state_dict()
    for k, v in sd.items():
        if "running" in k:
            assert torch.equal(v, fe.bufs.view("online_net." + k)), k
    for n, p in net.named_parameters():
        assert torch.equal(p.grad, fe.train.view("online_net." + n, fe.grad)), n


# ------------------------------------------------------------------------------------------ 4. BYOL in plain PyTorch
def test_plain_pytorch_byol_step_matches_the_fused_step():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL, R2Plus1DNet
    torch.manual_seed(0)
    m = R21DBYOL(pretrain=True)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    m.cuda().train()
    x1, x2 = _clips(seed=7), _clips(seed=8)
    labels = tuple(torch.randint(0, 5, (B,), device="cuda") for _ in range(5))
    fused = m.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=0.03)[7].item()

    def sub(prefix):
        return {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)}
    online, target = R2Plus1DNet(proj_flag=True), R2Plus1DNet(proj_flag=True)
    online.load_state_dict(sub("online_net."))
    tsd = sub("target_net.")
    with torch.no_grad():                     # R21DBYOL._update_target_net (r21d_byol.py:331-337) before the target calls
        for name, p in sub("online_net.").items():
            if not name.endswith(("running_mean", "running_var", "num_batches_tracked")):
                tsd[name] = tsd[name] * 0.996 + p * (1 - 0.996)
    target.load_state_dict(tsd)
    predictor = torch.nn.Sequential(torch.nn.Linear(512, 4096), torch.nn.BatchNorm1d(4096), torch.nn.ReLU(),
                                    torch.nn.Linear(4096, 512))
    predictor.load_state_dict({k[len("predictor.net."):]: v for k, v in sd.items() if k.startswith("predictor.net.")})
    online.cuda().train()
    target.cuda().train()
    predictor.cuda().train()

    def lf(a, b):
        return 2 - 2 * (F.normalize(a, dim=-1) * F.normalize(b, dim=-1)).sum(-1)
    _, p1 = online(x1)
    _, p2 = online(x2)
    q1, q2 = predictor(p1), predictor(p2)
    with torch.no_grad():
        _, t1 = target(x1)
        _, t2 = target(x2)
    loss = (lf(q1, t2) + lf(q2, t1)).mean()
    loss.backward()
    assert abs(loss.item() - fused) < 1e-3 * abs(fused), (loss.item(), fused)
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in online.parameters())


# ------------------------------------------------------------------------------------------ 5. input gradient kernel
@pytest.mark.parametrize("N,Tn,H,W", [(2, 4, 112, 112), (3, 2, 30, 100), (1, 3, 8, 4)])
def test_input_gradient_kernel_is_bit_exact_and_deterministic(N, Tn, H, W):
    from cstp_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(H + W)
    d = (torch.randn(N, Tn, H // 2, W // 2, 96, device="cuda", generator=g) * 1e-2).to(torch.bfloat16)
    d[..., 83:] = 0
    w = torch.randn(83, 3, 1, 7, 7, device="cuda", generator=g) * 0.05
    a = torch.full((N, 3, Tn, H, W), float("nan"), device="cuda")
    b = torch.empty_like(a)
    ops.stem_dgrad(d, w, a)
    ops.stem_dgrad(d, w, b)
    torch.cuda.synchronize()
    assert torch.equal(a, b)
    assert torch.equal(a.cpu(), stem_dgrad_reference(d.cpu(), w.cpu(), H, W))


def test_input_gradient_of_a_call_is_bit_exact_on_its_own_d_raw():
    net = _net(False)
    x = _clips(seed=9).requires_grad_(True)
    net(x).sum().backward()
    eng = _pooled(net, "grad")
    ref = stem_dgrad_reference(eng._stem_holder["g"].cpu(), eng.train.view("online_net.conv1.spatial_conv.weight").cpu(),
                               S, S)
    assert torch.equal(x.grad.cpu(), ref)


def test_input_gradient_wrapper_rejects_bad_arguments():
    from cstp_b200 import ops
    from cstp_b200.lib import CstpError
    d = torch.zeros(1, 2, 4, 4, 96, device="cuda", dtype=torch.bfloat16)
    w = torch.zeros(83, 3, 1, 7, 7, device="cuda")
    with pytest.raises(CstpError):
        ops.stem_dgrad(d, w, torch.zeros(1, 3, 2, 8, 10, device="cuda"))            # W not a multiple of 4
    with pytest.raises(CstpError):
        ops.stem_dgrad(d.float(), w, torch.zeros(1, 3, 2, 8, 8, device="cuda"))     # d(raw) not bf16
    with pytest.raises(CstpError):
        ops.stem_dgrad(d, w.cpu(), torch.zeros(1, 3, 2, 8, 8, device="cuda"))
    with pytest.raises(CstpError):
        ops.stem_dgrad(d, w, torch.zeros(1, 3, 2, 8, 8, device="cuda", dtype=torch.float64))


# ------------------------------------------------------------------------------------------ 6. optimiser and lifecycle
def _fresh_like(net, proj, grad, x):
    """The same call on a new module loaded with net's current state_dict (its engines are built and packed anew)."""
    fresh = _net(proj, seed=5)
    fresh.load_state_dict({k: v.clone() for k, v in net.state_dict().items()})
    if grad:
        return fresh(x)
    with torch.no_grad():
        return fresh(x)


def test_sgd_step_reaches_the_next_grad_call_on_the_pooled_engine():
    net = _net(True)
    x = _clips(seed=11)
    opt = torch.optim.SGD(net.parameters(), lr=0.05, momentum=0.9)
    for _ in range(2):
        f, p = net(x)
        (f.square().mean() + p.square().mean()).backward()
        opt.step()
        opt.zero_grad()
    assert len(net._pools[(B, T, S, S, torch.device("cuda", torch.cuda.current_device()), "grad")]) == 1
    want = _fresh_like(net, True, True, x)
    got = net(x)                                 # reuses the engine that was packed before the steps
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_in_place_target_update_reaches_the_next_no_grad_call():
    online, target = _net(True), _net(True, seed=4)
    x = _clips(seed=14)
    with torch.no_grad():
        target(x)
        for pt, po in zip(target.parameters(), online.parameters()):      # EMA in place (r21d_byol.py:331-337)
            pt.mul_(0.996).add_(po, alpha=0.004)
    want = _fresh_like(target, True, False, x)
    with torch.no_grad():
        got = target(x)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def test_memory_stays_flat_over_repeated_byol_calls():
    net = _net(True)
    opt = torch.optim.SGD(net.parameters(), lr=1e-3)
    x1, x2 = _clips(seed=12), _clips(seed=13).requires_grad_(True)
    mem = []
    for _ in range(50):
        f1, p1 = net(x1)
        f2, p2 = net(x2)
        (p1 * p2).sum().backward()
        opt.step()
        opt.zero_grad(set_to_none=False)
        x2.grad = None
        torch.cuda.synchronize()
        mem.append(torch.cuda.memory_allocated())
    assert len(mem) == 50 and len(set(mem[1:])) == 1, (mem[0], min(mem[1:]), max(mem[1:]))
    assert len(_pooled_all(net)) == 2
    # after 50 optimiser steps the pooled engines compute with the current weights
    want = _fresh_like(net, True, True, x1)
    got = net(x1)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


def _pooled_all(net):
    return [e for pool in net._pools.values() for e in pool]
