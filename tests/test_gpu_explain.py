"""Grad-CAM (cstp_b200.explain) on the B200: the three kernels of csrc/explain.cu and the eval-mode BatchNorm backward
bit-exact against their float32 stand-ins (tests/emulate_explain.py) on real engine buffers, logits bit-identical to the
model's eval forward, graph replay against the eager run, CAMs and the input gradient against fp32 torch autograd on the
same weights, and a finetune step unchanged by an explain call."""
import numpy as np
import pytest
import torch

from oracle import cstp_oracle as O
from tests import emulate_explain as EX
from tests.parity import rel
from tests.test_explain_cpu import reference_cam

pytestmark = pytest.mark.gpu

T, S = 16, 112
STAGES = ("conv2", "conv3", "conv4", "conv5")


def _np(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope="module")
def setup():
    """A finetune model on cuda:0 in eval mode and the structured clips it runs on.  Its running statistics are settled on
    those clips (the initial ones give near-zero features): the batch means, and the batch variances plus their mean over
    the layer's channels.  With the bare batch variances, channels of these smooth synthetic clips whose raw conv output
    has |mean| >> std turn the bf16 rounding of that output into large normalised errors, and the eval forward alone --
    the inference engines' program, unchanged here -- is 9.7e-2 off fp32 in its logits."""
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)
    settle = O.structured_batch(8, 0, T, S)[0].cuda()
    state = {k: v.cuda() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    with torch.no_grad():
        _, bufs = O.finetune_forward(state, settle, training=True)
    upd = {}
    for k, v in bufs.items():
        var = (v - 0.9) * 10
        upd[k] = (v * 10 if k.endswith("running_mean") else var + var.mean()).cpu()
    m.load_state_dict(upd, strict=False)
    m.cuda().eval()
    return m, settle


def _engine(m, n, stage, input_grad=False):
    from cstp_b200.engine_ft import inference_capacity
    return m._infer[("explain", inference_capacity(n), T, S, S, stage, input_grad, torch.device("cuda", 0))]


def test_kernels_bit_exact_on_engine_buffers(setup):
    from cstp_b200.explain import class_activation_maps
    m, x = setup
    n = 5
    for stage in STAGES:
        for classes in (None, torch.tensor([3, 100, 0, 7, 7])):
            r = class_activation_maps(m, x[:n], classes, stage=stage)
            torch.cuda.synchronize()
            eng = _engine(m, n, stage)
            k, d = EX.cam_seed_reference(_np(eng.logits), n, 101, None if classes is None else classes.numpy())
            assert np.array_equal(eng.classes.cpu().numpy(), k) and np.array_equal(_np(eng.dlogits), d)
            assert torch.equal(r.classes.cpu(), torch.from_numpy(k[:n]))
            alpha, cam = EX.gradcam_reference(_np(eng.stage_act[:n]), _np(eng.stage_grad[:n]), eng.stage_channels)
            assert np.array_equal(_np(eng.alpha[:n]), alpha), stage
            assert np.array_equal(_np(eng.cam_small[:n]), cam), stage
            up = EX.upsample_reference(_np(eng.cam_small[:n]), T, S, S)
            assert np.array_equal(_np(eng.cam[:n]), up) and np.array_equal(_np(r.cam), up), stage


def test_eval_batchnorm_backward_is_the_scaled_masked_gradient():
    from cstp_b200 import ops
    g = torch.Generator().manual_seed(4)
    rows, C, Cp = 4096, 83, 96
    st = ops.BNState.alloc(C, Cp, 1, rows, "cuda", eval_backward=True)
    gamma, beta = torch.randn(C, generator=g).cuda(), torch.randn(C, generator=g).cuda()
    rm, rv = torch.randn(C, generator=g).cuda(), (torch.rand(C, generator=g) + 0.5).cuda()
    ops.bn_eval_coeffs(st, gamma, beta, rm, rv)
    d = torch.randn(rows, Cp, generator=g).to(torch.bfloat16).cuda()
    raw = torch.randn(rows, Cp, generator=g).to(torch.bfloat16).cuda()
    act = torch.relu(torch.randn(rows, Cp, generator=g)).to(torch.bfloat16).cuda()
    scale = _np(st.scale)
    for mode in ("none", "act", "raw"):
        out, dz = torch.empty_like(d), torch.empty_like(d)
        ops.bn_backward_eval(d, act if mode == "act" else None, raw, st, out, dz=dz, mask_from_raw=mode == "raw")
        mask = None
        if mode == "act":
            mask = _np(act) > 0
        elif mode == "raw":    # the forward apply's fmaf, evaluated exactly in float64 (only its sign matters)
            mask = _np(raw).astype(np.float64) * scale + _np(st.shift).astype(np.float64) > 0
        ref = EX.bn_backward_eval_reference(_np(d), scale, mask)
        assert torch.equal(out.cpu(), torch.from_numpy(ref).to(torch.bfloat16)), mode
        assert torch.equal(dz.cpu().float(), torch.from_numpy(np.where(mask, _np(d), 0) if mask is not None else _np(d))), mode


@pytest.mark.parametrize("n", [1, 3, 7, 33, 70])
def test_logits_bit_identical_to_the_eval_forward(setup, n):
    from cstp_b200.explain import class_activation_maps
    m, x = setup
    xs = x.repeat(9, 1, 1, 1, 1)[:n] + torch.arange(n, device="cuda").view(-1, 1, 1, 1, 1) * 1e-3
    r = class_activation_maps(m, xs, stage="conv5")
    with torch.no_grad():
        ref = m(xs, o_type="test")
    assert torch.equal(r.logits, ref)
    assert torch.equal(r.classes, ref.argmax(1))
    assert r.cam.shape == (n, T, S, S)


def test_graph_replay_matches_the_eager_run(setup):
    from cstp_b200.explain import class_activation_maps
    m, x = setup
    runs = [class_activation_maps(m, x[:6], stage="conv3", input_grad=True) for _ in range(3)]   # eager, capture, replay
    eng = _engine(m, 6, "conv3", True)
    assert "explain" in eng._graphs
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert torch.equal(a, b)


# Relative L2 error bounds against fp32 autograd.  The project's bf16 bar is 1e-2 per tensor; logits and the conv5 map
# meet it (measured on a B200: 3.8e-3 and 4.7e-3).  The others do not, by the measured margins noted here, because a
# Grad-CAM map is relu(sum_c alpha_c A_c), a small difference of large terms of both signs that the min-max
# normalisation then stretches to [0, 1], so the 2^-9 relative rounding of bf16 activations and gradients is magnified;
# the input gradient crosses every bf16 dgrad of the network.  The emulated fp32 run of the same program
# (tests/test_explain_cpu.py) meets 1e-4 for every stage, so these margins are storage precision, not wiring.
BOUNDS = {"logits": 1e-2, "conv5": 1e-2,
          "conv3": 2.5e-2,          # measured 1.2e-2
          "conv4": 1.5e-1,          # measured 9.0e-2
          "conv2": 1.5e-1,          # measured 6.7e-2
          "input_grad": 4e-1}       # measured 2.0e-1


def test_against_fp32_autograd(setup, monkeypatch):
    """CAMs of every stage and the input gradient against the fp32 torch definition on the same weights (BOUNDS)."""
    from cstp_b200.explain import class_activation_maps
    m, x = setup
    state = {k: v for k, v in m.state_dict().items()}
    errs = {}
    for stage in STAGES:
        r = class_activation_maps(m, x, stage=stage, input_grad=stage == "conv2")
        lg, k, cam, dx = reference_cam(state, x, r.classes, stage, monkeypatch)
        errs[stage] = rel(r.cam, cam)
        errs["logits"] = rel(r.logits, lg)
        if stage == "conv2":
            errs["input_grad"] = rel(r.input_grad, dx)
        assert torch.equal(r.classes, lg.argmax(1))          # the explained class is fp32's prediction too
    print("relative L2 errors against fp32 autograd:", {k: f"{v:.2e}" for k, v in errs.items()})
    assert all(errs[k] < b for k, b in BOUNDS.items()), errs


def test_finetune_step_unchanged_by_an_explain_call(setup):
    from cstp_b200 import ops
    from cstp_b200.explain import class_activation_maps
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    _, x = setup
    labels = torch.tensor([3, 77, 5, 9], device="cuda")
    out = []
    for explain in (False, True):
        torch.manual_seed(1)
        m = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda()
        m.train()
        m.finetune_step(x[:4], labels)
        if explain:
            class_activation_maps(m, x[:3], stage="conv4", input_grad=True)
        torch.cuda.synchronize()
        n0 = ops.launch_count()
        loss = m.finetune_step(x[:4], labels).clone()
        torch.cuda.synchronize()
        out.append((loss, ops.launch_count() - n0, {k: v.clone() for k, v in m.state_dict().items()}))
    assert torch.equal(out[0][0], out[1][0]) and out[0][1] == out[1][1]
    assert all(torch.equal(v, out[1][2][k]) for k, v in out[0][2].items())
