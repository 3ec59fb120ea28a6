"""CPU stand-ins of the retrieval entry points (cstp_l2_normalize_rows / cstp_knn_partial / cstp_knn_merge) in numpy
float32, in the kernels' order of operations, so their results are the kernels' bits -- TEST INFRASTRUCTURE ONLY.  Every
other attribute resolves to tests/emulate_video_eval.py, so this module can stand in for `cstp_b200.ops` wherever the
feature-extraction and retrieval drivers run over the CPU emulator."""
from __future__ import annotations

import numpy as np
import torch

from cstp_b200.ops import knn_splits  # noqa: F401  (host-side choice, shared with the product path)
from tests import emulate_video_eval as _base
from tests.emulate_ops import _count

F32 = np.float32


def __getattr__(name):
    return getattr(_base, name)


def l2_normalize_rows(x, y):
    _count()
    d = y.shape[1]
    X = x[:, :d].detach().cpu().numpy().astype(F32)
    n = X.shape[0]
    lanes = np.zeros((n, 32), dtype=F32)                       # lane l adds columns l, l + 32, ... in order
    for j0 in range(0, d, 32):
        cols = X[:, j0:j0 + 32]
        lanes[:, :cols.shape[1]] = lanes[:, :cols.shape[1]] + cols * cols
    perm = np.arange(32)
    for o in (16, 8, 4, 2, 1):                                 # the xor butterfly: every lane ends with the same sum
        lanes = lanes + lanes[:, perm ^ o]
    nrm = np.maximum(np.sqrt(lanes[:, 0]), F32(1e-12))
    y.copy_(torch.from_numpy(X / nrm[:, None]))


def similarities(q, g):
    """s(q, g) for every pair: the chain acc + q[j] g[j] over j = 0 .. d-1, each product and sum rounded to fp32."""
    Q, G = q.detach().cpu().numpy().astype(F32), g.detach().cpu().numpy().astype(F32)
    acc = np.zeros((Q.shape[0], G.shape[0]), dtype=F32)
    for j in range(Q.shape[1]):
        acc += Q[:, j:j + 1] * G[None, :, j]
    return acc


def _top(vals, idx, k):
    """The first k of (vals, idx) by similarity descending, then the lower index; padded with -inf / -1."""
    order = np.lexsort((idx, -vals))[:k]
    v = np.full(k, -np.inf, dtype=F32)
    i = np.full(k, -1, dtype=np.int64)
    v[:len(order)], i[:len(order)] = vals[order], idx[order]
    return v, i


def knn_partial(q, g, k, splits, part_val, part_idx):
    _count()
    s = similarities(q, g)
    nq, ng = s.shape
    for sp in range(splits):
        lo, hi = ng * sp // splits, ng * (sp + 1) // splits
        for r in range(nq):
            v, i = _top(s[r, lo:hi], np.arange(lo, hi), k)
            part_val[sp, r] = torch.from_numpy(v)
            part_idx[sp, r] = torch.from_numpy(i.astype(np.int32))


def knn_merge(part_val, part_idx, idx_out, sim_out, q_labels=None, g_labels=None, cutoffs=None, hits=None):
    _count()
    splits, nq, k = part_val.shape
    pv, pi = part_val.numpy(), part_idx.numpy().astype(np.int64)
    for r in range(nq):
        keep = pi[:, r].reshape(-1) >= 0
        v, i = _top(pv[:, r].reshape(-1)[keep], pi[:, r].reshape(-1)[keep], k)
        idx_out[r] = torch.from_numpy(i)
        sim_out[r] = torch.from_numpy(v)
        if hits is not None:
            match = [j for j in range(k) if i[j] >= 0 and int(g_labels[i[j]]) == int(q_labels[r])]
            first = match[0] if match else k
            for c, cut in enumerate(cutoffs.tolist()):
                hits[c] += int(first < cut)
