"""Grad-CAM (cstp_b200.explain) on CPU: the float32 stand-ins of csrc/explain.cu against float64 torch, and
class_activation_maps through the emulated op layer (tests/emulate_explain.py, fp32 storage) against torch autograd on
the oracle's eval-mode finetune forward."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cstp_oracle as O
from tests import emulate_explain as EX
from tests.parity import rel

STAGE_RELU = {"conv2": 5, "conv3": 10, "conv4": 15, "conv5": 20}     # block outputs among the eval forward's 21 ReLUs
STAGE_CHANNELS = {"conv2": 64, "conv3": 128, "conv4": 256, "conv5": 512}


def _model():
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    return R21DBYOL(pretrain=False, num_classes=101, cls_bn=True)


def _settled(m, x):
    """Running statistics set to the batch statistics of x (one oracle training forward from mean 0 / var 1 with momentum
    0.1), so that the eval forward is far from its near-zero initial state."""
    state = {k: v.clone() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    with torch.no_grad():
        _, bufs = O.finetune_forward(state, x, training=True)
    upd = {k: (v * 10 if k.endswith("running_mean") else (v - 0.9) * 10) for k, v in bufs.items()}
    m.load_state_dict(upd, strict=False)
    return m


def reference_cam(state, x, classes, stage, monkeypatch):
    """The issue's definition in fp32 torch: (logits, classes, normalised cam, input gradient)."""
    seen = []

    class _Relu:
        def __getattr__(self, k):
            return getattr(F, k)

        @staticmethod
        def relu(t):
            seen.append(F.relu(t))
            return seen[-1]
    monkeypatch.setattr(O, "F", _Relu())
    x = x.clone().requires_grad_(True)
    logits, _ = O.finetune_forward(state, x, training=False)
    monkeypatch.undo()
    assert len(seen) == 21
    A = seen[STAGE_RELU[stage]]
    assert A.shape[1] == STAGE_CHANNELS[stage]
    k = classes if classes is not None else logits.argmax(1)
    score = logits.gather(1, k[:, None]).sum()
    dA, dx = torch.autograd.grad(score, [A, x])
    alpha = dA.mean(dim=(2, 3, 4))
    cam = F.relu((alpha[:, :, None, None, None] * A).sum(1))
    cam = F.interpolate(cam[:, None], size=x.shape[2:], mode="trilinear", align_corners=False)[:, 0]
    lo = cam.flatten(1).min(1).values[:, None, None, None]
    hi = cam.flatten(1).max(1).values[:, None, None, None]
    cam = torch.where(hi > lo, (cam - lo) / (hi - lo).clamp_min(1e-30), torch.zeros_like(cam))
    return logits.detach(), k, cam.detach(), dx


@pytest.fixture()
def emu():
    from cstp_b200 import engine
    saved = engine.ops, engine.ACT_DTYPE
    engine.ops, engine.ACT_DTYPE = EX, torch.float32
    try:
        yield engine
    finally:
        engine.ops, engine.ACT_DTYPE = saved


# ---------------------------------------------------------------------------------------------------- stand-ins
def test_gradcam_stand_in_matches_float64():
    g = torch.Generator().manual_seed(0)
    for (n, t, h, w, C, Cp) in ((2, 2, 7, 7, 512, 512), (3, 4, 5, 3, 24, 32), (1, 1, 1, 1, 8, 16)):
        act = torch.relu(torch.randn(n, t, h, w, Cp, generator=g)).to(torch.bfloat16).float()
        grad = (torch.randn(n, t, h, w, Cp, generator=g) * 1e-3).to(torch.bfloat16).float()
        alpha, cam = EX.gradcam_reference(act.numpy(), grad.numpy(), C)
        a64 = grad[..., :C].double().mean(dim=(1, 2, 3))
        c64 = torch.relu((a64[:, None, None, None, :] * act[..., :C].double()).sum(-1))
        assert rel(torch.from_numpy(alpha).double(), a64) < 1e-6
        assert rel(torch.from_numpy(cam).double(), c64) < 1e-5


def test_upsample_stand_in_matches_torch_trilinear_and_normalises():
    g = torch.Generator().manual_seed(1)
    for (t, h, w, T, H, W) in ((2, 7, 7, 16, 112, 112), (4, 14, 14, 16, 112, 112), (3, 5, 6, 8, 20, 12), (1, 1, 1, 4, 8, 8),
                               (5, 9, 7, 7, 9, 7)):
        cam = torch.rand(3, t, h, w, generator=g)
        cam[1] = 0.25                                                  # a flat map
        up = F.interpolate(cam[:, None].double(), size=(T, H, W), mode="trilinear", align_corners=False)[:, 0]
        got = EX.upsample_reference(cam.numpy(), T, H, W)
        for b in (0, 2):
            u = up[b]
            ref = (u - u.min()) / (u.max() - u.min()) if u.max() > u.min() else torch.zeros_like(u)
            assert rel(torch.from_numpy(got[b]).double(), ref) < 1e-6, (t, h, w, T, H, W)
        assert (got[1] == 0).all()
        assert got.min() >= 0 and got.max() <= 1


def test_seed_stand_in_argmax_ties_to_the_lower_class():
    lg = np.zeros((4, 16), np.float32)
    lg[0, [3, 7]] = 2.0
    lg[1, :5] = -1.0
    lg[1, 5:] = -3.0
    lg[2, 9] = 1.0
    lg[2, 12] = 5.0                         # a padding column: never chosen
    k, d = EX.cam_seed_reference(lg, 3, 10)
    assert k.tolist() == [3, 0, 9, 0]
    assert (d.sum(1) == [1, 1, 1, 0]).all() and d[0, 3] == 1 and d[3].sum() == 0
    k, d = EX.cam_seed_reference(lg, 2, 10, np.array([8, 1]))
    assert k.tolist() == [8, 1, 0, 0] and d[0, 8] == 1 and d[1, 1] == 1


def test_eval_backward_apply_stand_in():
    g = torch.Generator().manual_seed(2)
    d = torch.randn(64, 16, generator=g).to(torch.bfloat16).float().numpy()
    s = torch.randn(16, generator=g).numpy()
    y = EX.bn_backward_eval_reference(d, s, d > 0)
    assert np.array_equal(y, np.where(d > 0, s * d, 0).astype(np.float32))
    assert not np.signbit(y[y == 0]).any()                            # zero products are stored as +0


# ---------------------------------------------------------------------------------------------------- end to end
@pytest.mark.parametrize("stage", ["conv2", "conv3", "conv4", "conv5"])
def test_emulated_cams_match_autograd(emu, stage, monkeypatch):
    from cstp_b200.explain import class_activation_maps
    B, T, S = 3, 8, 32
    x = O.structured_batch(B, 0, T, S)[0]
    m = _settled(_model(), x).eval()
    state = {k: v.clone() for k, v in m.state_dict().items()}
    for classes in (None, torch.tensor([5, 0, 100])):
        r = class_activation_maps(m, x, classes, stage=stage, input_grad=stage == "conv2")
        lg, k, cam, dx = reference_cam(state, x, classes, stage, monkeypatch)
        assert r.logits.shape == (B, 101) and rel(r.logits, lg) < 1e-4
        assert torch.equal(r.classes, k)
        assert r.cam.shape == (B, T, S, S) and rel(r.cam, cam) < 1e-4, rel(r.cam, cam)
        if stage == "conv2":
            # the stem input gradient rounds the stem weight to bf16, as the packed weights of every dgrad are
            assert r.input_grad.shape == x.shape and rel(r.input_grad, dx) < 1e-2
        else:
            assert r.input_grad is None


@pytest.mark.parametrize("n", [1, 3, 70])
def test_emulated_chunking(emu, n, monkeypatch):
    from cstp_b200.explain import class_activation_maps
    T, S = 8, 32
    x = O.structured_batch(n, 2, T, S)[0]
    m = _settled(_model(), O.structured_batch(4, 0, T, S)[0])
    state = {k: v.clone() for k, v in m.state_dict().items()}
    r = class_activation_maps(m, x, stage="conv3")
    lg, k, cam, _ = reference_cam(state, x, None, "conv3", monkeypatch)
    assert r.cam.shape == (n, T, S, S) and torch.equal(r.classes, k)
    # the per-clip min-max normalisation magnifies fp32 rounding where a clip's map spans a small range
    assert rel(r.logits, lg) < 1e-4 and rel(r.cam, cam) < 1e-2


def test_emulated_call_changes_nothing(emu):
    from cstp_b200.explain import class_activation_maps
    x = O.structured_batch(2, 1, 4, 32)[0]
    m = _settled(_model(), x)
    m.train()                                   # eval semantics regardless of the mode
    before = {k: v.clone() for k, v in m.state_dict().items()}
    rng = torch.get_rng_state()
    a = class_activation_maps(m, x, stage="conv3", input_grad=True)
    assert m.training
    after = m.state_dict()
    assert before.keys() == after.keys() and all(torch.equal(before[k], after[k]) for k in before)
    assert torch.equal(rng, torch.get_rng_state())
    m.eval()
    b = class_activation_maps(m, x, stage="conv3", input_grad=True)
    assert torch.equal(a.cam, b.cam) and torch.equal(a.logits, b.logits) and torch.equal(a.input_grad, b.input_grad)
    assert any(k[0] == "explain" for k in m._infer)
    m.free_inference_engines()
    assert not m._infer


def test_rejections(emu):
    from cstp_b200.explain import class_activation_maps
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    m = _model()
    x = torch.zeros(2, 3, 4, 16, 16)
    with pytest.raises(ValueError, match="finetune model"):
        class_activation_maps(R21DBYOL(pretrain=True), x)
    with pytest.raises(ValueError, match="finetune model"):
        class_activation_maps(torch.nn.Linear(2, 2), x)
    with pytest.raises(ValueError, match="stage"):
        class_activation_maps(m, x, stage="conv1")
    with pytest.raises(ValueError, match="n, 3, T, H, W"):
        class_activation_maps(m, x[0])
    with pytest.raises(ValueError, match="n, 3, T, H, W"):
        class_activation_maps(m, x[:, :2])
    with pytest.raises(TypeError, match="float32"):
        class_activation_maps(m, x.double())
    with pytest.raises(ValueError, match="stem"):
        class_activation_maps(m, torch.zeros(2, 3, 4, 15, 16))
    with pytest.raises(ValueError, match="stem"):
        class_activation_maps(m, torch.zeros(2, 3, 4, 16, 18))
    with pytest.raises(ValueError, match="one integer class per clip"):
        class_activation_maps(m, x, [1])
    with pytest.raises(ValueError, match="one integer class per clip"):
        class_activation_maps(m, x, torch.tensor([1.0, 2.0]))
    with pytest.raises(ValueError, match=r"\[0, 101\)"):
        class_activation_maps(m, x, [0, 101])
    with pytest.raises(ValueError, match=r"\[0, 101\)"):
        class_activation_maps(m, x, [-1, 3])


def test_cpu_clips_are_rejected_by_the_device_path():
    from cstp_b200 import lib as L
    from cstp_b200.explain import class_activation_maps
    with pytest.raises(L.CstpError, match="CUDA"):
        class_activation_maps(_model(), torch.zeros(1, 3, 4, 16, 16))
