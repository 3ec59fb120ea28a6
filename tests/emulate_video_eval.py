"""CPU stand-ins of the video-level scoring entry points (cstp_video_accumulate / cstp_video_finalize) -- TEST
INFRASTRUCTURE ONLY.  Every other attribute resolves to tests/emulate_ops.py, so this module can stand in for
`cstp_b200.ops` wherever the engine and the test-evaluation driver run over the CPU emulator."""
from __future__ import annotations

import torch

from tests import emulate_ops as _base
from tests.emulate_ops import _count


def __getattr__(name):
    return getattr(_base, name)


def video_accumulate(logits, n_cls, seg, sums, rows=None):
    _count()
    rows = rows or logits.shape[0]
    for slot, first, count in seg.tolist():
        if count <= 0 or not 0 <= slot < sums.shape[0] or first < 0 or first + count > rows:
            continue
        acc = sums[slot].clone()
        for r in range(first, first + count):                # clip order, one fp32 rounding per addition
            acc += logits[r, :n_cls]
        sums[slot] = acc


def video_finalize(sums, fin, topk_out, labels=None, mean_out=None, hits=None):
    _count()
    n_cls, k = sums.shape[1], topk_out.shape[1]
    for slot, count, video in fin.tolist():
        if count <= 0 or not 0 <= slot < sums.shape[0] or not 0 <= video < topk_out.shape[0]:
            continue
        mean = sums[slot] / float(count)
        # descending by value, ties to the lower class index
        order = sorted(range(n_cls), key=lambda c: (-mean[c].item(), c))[:max(k, 5)]
        topk_out[video] = torch.tensor([order[j] if j < len(order) else -1 for j in range(k)], dtype=topk_out.dtype)
        if hits is not None:
            y = int(labels[video])
            hits[0] += int(order[0] == y)
            hits[1] += int(y in order[:5])
        if mean_out is not None:
            mean_out[video] = mean
        sums[slot] = 0
