"""Float32 stand-in of cstp_repr_stats (csrc/loss_optim.cu) -- TEST INFRASTRUCTURE ONLY.

`repr_stats_np` restates the kernel in numpy float32, one correctly rounded operation at a time and in the kernel's order
(numpy does not contract a * b + c into an FMA, and every sum here is an explicit loop, never np.sum), so it reproduces
the kernel's bits.  `repr_stats` has the signature of cstp_b200.ops.repr_stats (and its argument checks) and runs on CPU
tensors; `install` adds it to tests/emulate_ops.py for the duration of one test."""
from __future__ import annotations

import numpy as np
import torch

F32 = np.float32
D = 512


def _row_norms(X: np.ndarray) -> np.ndarray:
    """||x_r||: lane l of a warp adds x[l]^2, x[l + 32]^2, ... in order, then the xor butterfly over 16, 8, 4, 2, 1."""
    lanes = np.zeros((X.shape[0], 32), dtype=F32)
    for j0 in range(0, D, 32):
        cols = X[:, j0:j0 + 32]
        lanes = lanes + cols * cols
    perm = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        lanes = lanes + lanes[:, perm ^ o]
    return np.sqrt(lanes[:, 0])


def view_stats(X: np.ndarray):
    """(s, mean row norm) of one view's rows X float32 [B][>= 512]."""
    X = np.ascontiguousarray(X[:, :D], dtype=F32)
    B = X.shape[0]
    n = _row_norms(X)
    z = X / np.maximum(n, F32(1e-12))[:, None]
    s1 = np.zeros(D, dtype=F32)
    for r in range(B):
        s1 = s1 + (z[r] - z[0])
    m = s1 / F32(B)
    s2 = np.zeros(D, dtype=F32)
    for r in range(B):
        d = (z[r] - z[0]) - m
        s2 = s2 + d * d
    a = np.sqrt(s2 / F32(B - 1))
    while a.shape[0] > 1:                       # red[t] += red[t + h] for h = 256, ..., 1
        h = a.shape[0] // 2
        a = a[:h] + a[h:]
    ns = F32(0)
    for r in range(B):
        ns = F32(ns + n[r])
    return F32(a[0] / F32(D)), F32(ns / F32(B))


def repr_stats_np(blocks, B: int) -> np.ndarray:
    """float32 [2][5] of cstp_repr_stats for blocks (feat, proj, pred, tproj), each [2B][>= 512] or None."""
    out = np.zeros((2, 5), dtype=F32)
    for k, x in enumerate(blocks):
        if x is None:
            continue
        X = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
        for v in range(2):
            s, nm = view_stats(X[v * B:(v + 1) * B])
            out[v, k] = s
            if k == 0:
                out[v, 4] = nm
    return out


def repr_stats(feat, proj, pred, tproj, B, out):
    from cstp_b200 import ops
    from tests import emulate_ops
    ops._check_repr_stats((feat, proj, pred, tproj), B, out)
    emulate_ops._count()
    out.view(-1)[:10].copy_(torch.from_numpy(repr_stats_np((feat, proj, pred, tproj), B).reshape(-1)))


def install(monkeypatch) -> None:
    from tests import emulate_ops
    monkeypatch.setattr(emulate_ops, "repr_stats", repr_stats, raising=False)


def float64_reference(x: torch.Tensor, B: int) -> torch.Tensor:
    """The definition in float64 torch: per view, mean_j of the unbiased std over rows of F.normalize(x)[:, j], and the
    mean row norm.  Returns [2][2] = (s, mean norm) per view."""
    x = x[:, :D].double()
    res = []
    for v in range(2):
        xv = x[v * B:(v + 1) * B]
        z = torch.nn.functional.normalize(xv, dim=1, eps=1e-12)
        res.append([z.std(dim=0, unbiased=True).mean().item(), xv.norm(dim=1).mean().item()])
    return torch.tensor(res, dtype=torch.float64)
