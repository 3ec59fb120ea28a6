"""CPU stand-in op layer of the standalone backbone -- TEST INFRASTRUCTURE ONLY.

Everything of tests/emulate_ops.py, plus `stem_dgrad`, the stem's input gradient (csrc/stem_dgrad.cu) restated in
numpy float32 in the kernel's summation order: channel pairs ascending, then kh, then kw, then the two channels of the
pair, each term one rounded addition of an exact product (both factors are bf16 values).  It reproduces the kernel's
bits.  Tests inject this module with monkeypatch in place of cstp_b200.ops.
"""
from __future__ import annotations

import numpy as np
import torch

from tests.emulate_ops import *  # noqa: F401,F403
from tests.emulate_ops import _count


def _bf16(t: torch.Tensor) -> np.ndarray:
    return t.detach().to(torch.bfloat16).float().cpu().numpy()


def stem_dgrad_reference(g: torch.Tensor, w: torch.Tensor, H: int, W: int) -> torch.Tensor:
    """g (N, T, H/2, W/2, Cg) -> fp32 (N, 3, T, H, W) in the kernel's order; the weight is rounded to bf16."""
    N, T, Ho, Wo, _ = g.shape
    cout = w.shape[0]
    gn = g.detach().float().cpu().numpy()[..., :cout].astype(np.float32)
    wn = _bf16(w.reshape(cout, 3, 7, 7))
    pairs = (cout + 1) // 2
    if cout % 2:
        gn = np.concatenate([gn, np.zeros(gn.shape[:-1] + (1,), np.float32)], -1)
        wn = np.concatenate([wn, np.zeros((1, 3, 7, 7), np.float32)], 0)
    # zero border of 3 d(raw) positions on every side: oh = (h + 3 - kh) / 2 ranges over [-1, Ho + 1]
    gp = np.zeros((N, T, Ho + 6, Wo + 6, 2 * pairs), np.float32)
    gp[:, :, 3:3 + Ho, 3:3 + Wo] = gn
    out = np.zeros((N, 3, T, H, W), np.float32)
    for hp in (0, 1):
        khs = [k for k in range(7) if (hp + 3 - k) % 2 == 0]
        for wp in (0, 1):
            kws = [k for k in range(7) if (wp + 3 - k) % 2 == 0]
            hs, ws = np.arange(hp, H, 2), np.arange(wp, W, 2)
            acc = np.zeros((3, N, T, len(hs), len(ws)), np.float32)
            for p in range(pairs):
                for kh in khs:
                    oh = (hs + 3 - kh) // 2 + 3
                    for kw in kws:
                        ow = (ws + 3 - kw) // 2 + 3
                        for co in (2 * p, 2 * p + 1):
                            gv = gp[:, :, oh][:, :, :, ow, co]                  # (N, T, |hs|, |ws|)
                            for c in range(3):
                                acc[c] = acc[c] + gv * wn[co, c, kh, kw]
            out[:, :, :, hp::2, wp::2] = acc.transpose(1, 0, 2, 3, 4)
    return torch.from_numpy(out)


def stem_dgrad(g, w, dx):
    _count()
    N, _, T, H, W = dx.shape
    dx.copy_(stem_dgrad_reference(g, w, H, W).to(dx.device))
