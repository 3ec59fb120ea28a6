"""Float32 stand-in of cstp_adam_clip_step / cstp_adam_clip_step_dev (csrc/loss_optim.cu) -- TEST INFRASTRUCTURE ONLY.

`adam_update` restates the kernel's per-element arithmetic in numpy float32, one correctly rounded operation at a time
(numpy does not contract a * b + c into an FMA), so it reproduces the kernel's bits for a given clip coefficient.
`adam_clip_step` / `adam_clip_step_dev` have the signatures of cstp_b200.ops and run the whole step on CPU tensors; the
gradient norm is summed in double (the kernel sums fp32 partials in a fixed order, so norms agree to rounding, not to
the bit).  `install` adds them to tests/emulate_ops.py for the duration of one test."""
from __future__ import annotations

import numpy as np
import torch

F32 = np.float32


def clip_coefficient(norm: float, max_norm: float, clip: bool) -> np.float32:
    """max_norm / (norm + 1e-6) capped at 1, in fp32 as the kernel computes it."""
    if not clip:
        return F32(1.0)
    c = F32(max_norm) / (F32(norm) + F32(1e-6))
    return min(c, F32(1.0))


def adam_update(p: np.ndarray, g: np.ndarray, m: np.ndarray, v: np.ndarray, coef, hyper) -> None:
    """One Adam / AdamW step in place on float32 arrays; hyper: the ten cstp_adam_hyper scalars in field order."""
    step_size, bc2_sqrt, omb1, beta2, omb2, eps, l2, decay = (F32(x) for x in hyper[:8])
    gr = g * F32(coef)
    p *= decay
    gr = gr + l2 * p
    m += (gr - m) * omb1
    v[...] = v * beta2 + (omb2 * gr) * gr
    den = np.sqrt(v) / bc2_sqrt + eps
    p -= (step_size * m) / den


def adam_clip_step(p, g, m, v, hyper, norm_out, workspace):
    from tests import emulate_ops
    emulate_ops._count(2)
    norm = F32(g.double().pow(2).sum().sqrt().item())
    coef = clip_coefficient(norm, hyper[8], hyper[9] != 0)
    adam_update(p.numpy(), g.numpy(), m.numpy(), v.numpy(), coef, hyper)
    norm_out[0], norm_out[1] = float(norm), float(coef)


def adam_clip_step_dev(p, g, m, v, hyper, norm_out, workspace):
    adam_clip_step(p, g, m, v, [float(x) for x in hyper.tolist()], norm_out, workspace)


def install(monkeypatch) -> None:
    from tests import emulate_ops
    monkeypatch.setattr(emulate_ops, "adam_clip_step", adam_clip_step, raising=False)
    monkeypatch.setattr(emulate_ops, "adam_clip_step_dev", adam_clip_step_dev, raising=False)


def torch_reference(params, grad_stream, kind, lr, betas, eps, wd, max_norm=None, device="cpu"):
    """torch.optim.Adam / AdamW (foreach=False) over `params` (list of fp32 tensors) fed grad_stream (list per step of
    lists of gradients), with clip_grad_norm_(max_norm) first when max_norm is set.  Returns (params, exp_avg,
    exp_avg_sq) after the last step."""
    ps = [torch.nn.Parameter(t.clone().to(device)) for t in params]
    cls = torch.optim.AdamW if kind == "adamw" else torch.optim.Adam
    opt = cls(ps, lr=lr, betas=betas, eps=eps, weight_decay=wd, foreach=False)
    for grads in grad_stream:
        for q, gr in zip(ps, grads):
            q.grad = None if gr is None else gr.clone().to(device)
        if max_norm is not None:
            torch.nn.utils.clip_grad_norm_([q for q in ps if q.grad is not None], max_norm)
        opt.step()
    st = [opt.state.get(q, {}) for q in ps]
    return ([q.detach().cpu() for q in ps], [s["exp_avg"].cpu() if s else None for s in st],
            [s["exp_avg_sq"].cpu() if s else None for s in st])
