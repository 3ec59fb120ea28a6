"""Nearest-neighbour video retrieval on one B200: per-video feature extraction (cstp_b200.evaluate.video_features) on the
seeded synthetic test set of tools/test_eval_bench.py, and the exact fp32 similarity + top-k kernels (csrc/retrieval.cu)
at two protocol sizes against torch fp32 `(q @ g.T).topk(k)` (TF32 off) on the same GPU.

    python tools/retrieval_bench.py [--out profiles/r04_retrieval_bench.json]

Sizes (seeded random 512-d features, k = 50): UCF101 split 1 test x train (3,783 x 9,537; its 19.5 MB gallery stays in
L2 between calls) and Kinetics-400 val x train (19,715 x 239,429; a 490 MB gallery, larger than L2).  Kernel times are
CUDA-event means over at least 1 s of timed calls after a warm-up; FLOP counts a multiply and an add per feature
element of every pair.  The line also says whether the baseline's recall@{1, 5, 10, 20, 50} agrees with the kernels' and
how many queries have a different top-50 set (the baseline's TF32-free GEMM rounds differently, so near-ties can swap).
Prints one JSON line and writes the same line to --out."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.test_eval_bench import CAPACITY, card, model, synthetic_set  # noqa: E402

K, D, KS = 50, 512, (1, 5, 10, 20, 50)
SIZES = {"ucf101_split1": (3783, 9537, 101), "kinetics400_val_train": (19715, 239429, 400)}
MIN_TIMED_S = 1.0
CHUNK_ELEMS = 1 << 30                     # baseline: rows of q @ g.T per chunk, at most 4 GB of fp32 similarities


def timed(fn, warm=2):
    """Mean ms per call of fn over at least MIN_TIMED_S of back-to-back calls (CUDA events), after `warm` calls."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    calls, total = 0, 0.0
    while total < MIN_TIMED_S * 1e3:
        n = max(1, calls)                 # 1, 1, 2, 4, ... calls per window
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        e1.synchronize()
        total += e0.elapsed_time(e1)
        calls += n
    return total / calls, calls


def kernel_search(qn, gn, ql, gl):
    from cstp_b200 import ops
    nq, ng = qn.shape[0], gn.shape[0]
    splits = ops.knn_splits(nq, ng)
    pv = torch.empty(splits, nq, K, device="cuda")
    pi = torch.empty(splits, nq, K, dtype=torch.int32, device="cuda")
    idx = torch.empty(nq, K, dtype=torch.int64, device="cuda")
    sim = torch.empty(nq, K, device="cuda")
    hits = torch.zeros(len(KS), dtype=torch.int64, device="cuda")
    cut = torch.tensor(KS, dtype=torch.int32, device="cuda")

    def run():
        hits.zero_()
        ops.knn_partial(qn, gn, K, splits, pv, pi)
        ops.knn_merge(pv, pi, idx, sim, ql, gl, cut, hits)
    return run, idx, hits, splits


def torch_search(qn, gn):
    rows = max(1, CHUNK_ELEMS // gn.shape[0])
    idx = torch.empty(qn.shape[0], K, dtype=torch.int64, device="cuda")

    def run():
        for r0 in range(0, qn.shape[0], rows):
            idx[r0:r0 + rows] = (qn[r0:r0 + rows] @ gn.T).topk(K, dim=1).indices
    return run, idx, rows


def recall_hits(idx, ql, gl):
    match = gl[idx] == ql[:, None]
    return [int(match[:, :c].any(1).sum()) for c in KS]


def knn_size(name, nq, ng, n_cls):
    from cstp_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(1)
    q = torch.randn(nq, D, device="cuda", generator=g)
    gal = torch.randn(ng, D, device="cuda", generator=g)
    ql = torch.randint(0, n_cls, (nq,), device="cuda", generator=g)
    gl = torch.randint(0, n_cls, (ng,), device="cuda", generator=g)
    qn, gn = torch.empty_like(q), torch.empty_like(gal)
    ops.l2_normalize_rows(q, qn)
    ops.l2_normalize_rows(gal, gn)
    flop = 2.0 * nq * ng * D
    run, idx, hits, splits = kernel_search(qn, gn, ql, gl)
    t_k, calls_k = timed(run)
    run()
    k_hits = hits.cpu().tolist()
    assert k_hits == recall_hits(idx, ql, gl)
    brun, bidx, rows = torch_search(qn, gn)
    t_b, calls_b = timed(brun)
    b_hits = recall_hits(bidx, ql, gl)
    differ = int((idx.sort(1).values != bidx.sort(1).values).any(1).sum())
    del q, gal
    return {"queries": nq, "gallery": ng, "d": D, "k": K, "gflop": flop / 1e9, "splits": splits,
            "kernel_ms": t_k, "kernel_calls_timed": calls_k, "kernel_tflops": flop / t_k / 1e9,
            "kernel_hits": dict(zip(map(str, KS), k_hits)),
            "torch_fp32_ms": t_b, "torch_calls_timed": calls_b, "torch_tflops": flop / t_b / 1e9,
            "torch_chunk_rows": rows, "torch_hits": dict(zip(map(str, KS), b_hits)),
            "recall_agrees_with_torch": k_hits == b_hits, "queries_with_different_top50_set": differ,
            "kernel_over_torch_time": t_k / t_b}


def features_rate():
    from cstp_b200.evaluate import video_features
    store, frames, _ = synthetic_set()
    m = model()
    video_features(m, store, frames, capacity=CAPACITY)           # builds the engine and captures its graph
    times = []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        f = video_features(m, store, frames, capacity=CAPACITY)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    from cstp_b200.data_process.clip_plan import FinetuneClipSampler
    sampler = FinetuneClipSampler(16, 112, 4)
    clips = sum(len(sampler.plan_test(n, store[v].shape[2], store[v].shape[1])) for v, n in enumerate(frames))
    t = sorted(times)[1]
    return {"videos": len(frames), "clips": clips, "capacity": CAPACITY, "pass_s": times, "videos_per_s": len(frames) / t,
            "clips_per_s": clips / t, "features_finite": bool(torch.isfinite(f).all())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_retrieval_bench.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("retrieval_bench measures on a CUDA device; none is visible")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    torch.set_float32_matmul_precision("highest")
    out = {**card(), "video_features": features_rate()}
    torch.cuda.empty_cache()
    for name, (nq, ng, n_cls) in SIZES.items():
        out[name] = knn_size(name, nq, ng, n_cls)
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
