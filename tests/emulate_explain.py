"""CPU stand-in op layer of the Grad-CAM path -- TEST INFRASTRUCTURE ONLY.

Everything of tests/emulate_backbone.py (tests/emulate_ops.py plus the stem's input gradient), plus numpy float32
restatements of the three kernels of csrc/explain.cu in their exact operation order -- cam_seed, gradcam (the position
sum in eight interleaved lanes, then lane order; rounded products added in channel order) and cam_upsample (torch's
align_corners=False source index, the w / h / t blends a + l * (b - a), per-clip min-max) -- and of the eval-mode use of the BatchNorm
backward apply (ops.bn_backward_eval: g = bf16(scale * dy), a zero product stored as +0).  numpy's float32 +, -, * and /
are correctly rounded, so these reproduce the kernels' bits.  Tests inject this module with monkeypatch in place of
cstp_b200.ops.
"""
from __future__ import annotations

import numpy as np
import torch

from tests.emulate_backbone import *  # noqa: F401,F403
from tests.emulate_ops import _count, _group_view

F32 = np.float32


def _np(t: torch.Tensor) -> np.ndarray:
    return t.detach().float().cpu().numpy().astype(F32)


def cam_seed_reference(logits: np.ndarray, n: int, n_cls: int, classes_in=None):
    """logits fp32 [B][ld] -> (classes int64 [B], dlogits fp32 [B][ld])."""
    B, ld = logits.shape
    k = np.zeros(B, np.int64)
    k[:n] = np.asarray(classes_in)[:n] if classes_in is not None else np.argmax(logits[:n, :n_cls], 1)
    d = np.zeros((B, ld), F32)
    d[np.arange(n), k[:n]] = 1.0
    return k, d


def gradcam_reference(act: np.ndarray, grad: np.ndarray, C: int):
    """act, grad (n, t, h, w, Cp) -> (alpha fp32 [n][C], cam fp32 (n, t, h, w))."""
    n, t, h, w, Cp = act.shape
    P = t * h * w
    d = grad.reshape(n, P, Cp)[:, :, :C].astype(F32)
    d = np.concatenate([d, np.zeros((n, (-P) % 8, C), F32)], 1).reshape(n, -1, 8, C)
    acc = np.zeros((n, 8, C), F32)
    for i in range(d.shape[1]):
        acc = acc + d[:, i]
    s = acc[:, 0]
    for q in range(1, 8):
        s = s + acc[:, q]
    alpha = s / F32(P)
    a = act.reshape(n, P, Cp)[:, :, :C].astype(F32)
    cam = np.zeros((n, P), F32)
    for c in range(C):
        cam = cam + alpha[:, c:c + 1] * a[:, :, c]
    cam = np.where(cam > 0, cam, F32(0))
    return alpha, cam.reshape(n, t, h, w)


def _axis(out: int, inn: int):
    scale = F32(inn) / F32(out)
    src = scale * (np.arange(out, dtype=F32) + F32(0.5)) - F32(0.5)
    src = np.where(src < 0, F32(0), src).astype(F32)
    i0 = src.astype(np.int64)
    i1 = i0 + (i0 < inn - 1)
    return i0, i1, (src - i0.astype(F32)).astype(F32)


def upsample_reference(cam: np.ndarray, T: int, H: int, W: int) -> np.ndarray:
    """cam fp32 (n, t, h, w) -> trilinear to (n, T, H, W), then per-clip (v - min) / (max - min), zeros when flat."""
    n, t, h, w = cam.shape
    t0, t1, lt = _axis(T, t)
    h0, h1, lh = _axis(H, h)
    w0, w1, lw = _axis(W, w)

    def mix(a, l, b):
        return a + l * (b - a)
    x = cam.astype(F32)
    xw = mix(x[..., w0], lw, x[..., w1])                                      # (n, t, h, W)
    xh = mix(xw[:, :, h0, :], lh[:, None], xw[:, :, h1, :])                   # (n, t, H, W)
    v = mix(xh[:, t0], lt[:, None, None], xh[:, t1])                          # (n, T, H, W)
    out = np.zeros_like(v)
    for b in range(n):
        mn, mx = v[b].min(), v[b].max()
        if mx > mn:
            out[b] = (v[b] - mn) / (mx - mn)
    return out


def bn_backward_eval_reference(d: np.ndarray, scale: np.ndarray, mask=None) -> np.ndarray:
    """fp32 g (before the bf16 store) of ops.bn_backward_eval: scale * (masked d), a zero product as +0."""
    dy = d if mask is None else np.where(mask, d, F32(0))
    return (scale.astype(F32) * dy + F32(0)).astype(F32)


# ---------------------------------------------------------------------------------------------------- ops layer
def bn_backward_eval(d, act, raw, st, g_out, *, dz=None, mask_from_raw=False):
    _count()
    Cp = st.Cp
    dy = _group_view(d, 1).float()
    if mask_from_raw:
        dy = dy * ((_group_view(raw, 1).float() * st.scale.view(1, 1, Cp) + st.shift.view(1, 1, Cp)) > 0)
    elif act is not None:
        dy = dy * (_group_view(act, 1).float() > 0)
    if dz is not None:
        dz.copy_(dy.reshape(dz.shape).to(dz.dtype))
    g = st.scale.view(1, 1, Cp) * dy + 0.0
    g_out.copy_(g.reshape(g_out.shape).to(g_out.dtype))


def cam_seed(logits, n, n_cls, classes_in, classes_out, dlogits):
    _count()
    k, d = cam_seed_reference(_np(logits), n, n_cls, None if classes_in is None else classes_in.cpu().numpy())
    classes_out.copy_(torch.from_numpy(k))
    dlogits.copy_(torch.from_numpy(d))


def gradcam(act, grad, n, C_, alpha, cam):
    _count(2)
    a, c = gradcam_reference(_np(act[:n]), _np(grad[:n]), C_)
    alpha.view(-1)[:a.size].copy_(torch.from_numpy(a).reshape(-1))
    cam.view(-1)[:c.size].copy_(torch.from_numpy(c).reshape(-1))


def cam_upsample(cam, n, out):
    _count()
    _, T, H, W = out.shape
    out[:n].copy_(torch.from_numpy(upsample_reference(_np(cam[:n]), T, H, W)))
