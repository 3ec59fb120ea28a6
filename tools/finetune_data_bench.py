"""Finetuning and test evaluation fed from JPEG frames against the same work fed from a resident store of decoded frames,
alternated in one run, on synthetic UCF101-sized videos (171x128, 4:2:0, quality 90, 100-272 frames, about 186 on
average as in UCF101):
  finetune   samples/s of `train.finetune_epochs` training epochs at batch 60, `JpegFinetuneBatches` vs `FinetuneBatches`
  test       videos/s of `evaluate.test_videos_jpeg` vs `evaluate.test_videos` (capacity 60), with results compared
The JPEG bytes are held in host memory, so read_frames costs no file-system time; a reader from disk adds its own.
    python tools/finetune_data_bench.py [out.json]"""
import io
import json
import os
import random
import subprocess
import sys
import time
import types
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cstp_b200 import train  # noqa: E402
from cstp_b200.data_process.datasets import FinetuneBatches, GpuVideoStore, JpegFinetuneBatches  # noqa: E402
from cstp_b200.evaluate import test_videos, test_videos_jpeg  # noqa: E402
from cstp_b200.models.pace.r21d_byol import R21DBYOL  # noqa: E402
from cstp_b200.synthetic import synthetic_video  # noqa: E402

W, H = 171, 128


def encode_video(args):
    n, seed = args
    out = []
    for f in synthetic_video(n, W, H, seed):
        b = io.BytesIO()
        Image.fromarray(f).save(b, "JPEG", quality=90, subsampling=2)
        out.append(b.getvalue())
    return out


def gpu_state():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    return q[0] if q else None


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else None
    res = {"gpu_before": gpu_state(), "host_cores": os.cpu_count()}
    rng = np.random.default_rng(0)
    n_train, n_test = 600, 240
    counts = [int(c) for c in rng.integers(100, 273, n_train + n_test)]
    t0 = time.perf_counter()
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        enc = list(ex.map(encode_video, [(n, v) for v, n in enumerate(counts)]))
    res["encode_s"] = time.perf_counter() - t0
    store = GpuVideoStore("cuda")
    for v, streams in enumerate(enc):
        store.put_jpeg(v, streams)
    labels = [v % 101 for v in range(n_train + n_test)]

    def read_frames(video, numbers):
        return [enc[video][k - 1] for k in numbers]

    def read_test(video, numbers):
        return read_frames(n_train + video, numbers)
    test_store = GpuVideoStore("cuda")
    for v in range(n_test):
        test_store.put(v, store[n_train + v])
    res["setup"] = {"train_videos": n_train, "test_videos": n_test, "size": [W, H], "mean_frames": float(np.mean(counts)),
                    "mean_bytes_per_frame": float(np.mean([len(b) for e in enc for b in e])), "batch": 60,
                    "store_GB": store.bytes / 1e9}

    # ---- finetune: training epochs through finetune_epochs (validation left out: an empty val source)
    torch.manual_seed(1)
    model = R21DBYOL(pretrain=False, num_classes=101, cls_bn=True).cuda()
    opts = types.SimpleNamespace(n_epochs=1, learning_rate=0.025, momentum=0.9, weight_decay=1e-3, lr_patience=10,
                                 task="ft_all")
    sources = {"jpeg": JpegFinetuneBatches(read_frames, counts[:n_train], labels[:n_train], 60),
               "store": FinetuneBatches(store, counts[:n_train], labels[:n_train], 60)}
    steps = n_train // 60

    def epoch(name, e):
        opts.n_epochs = e
        rows, _ = train.finetune_epochs(model, sources[name], lambda _: iter(()), opts, begin_epoch=e)
        return rows
    random.seed(0)
    for name in sources:                                 # warm-up: engine, graphs, staging buffers
        epoch(name, 1)
    ft = {k: [] for k in sources}
    rounds = 8
    for r in range(rounds):
        for name in (("jpeg", "store") if r % 2 == 0 else ("store", "jpeg")):
            dt, rows = timed(lambda: epoch(name, r + 2))
            assert np.isfinite(rows[0]["loss"])
            ft[name].append(steps * 60 / dt)
    res["finetune_b60"] = {k: {"samples_per_s_median": float(np.median(v)), "per_round": v} for k, v in ft.items()}
    res["finetune_b60"]["jpeg_over_store"] = (res["finetune_b60"]["jpeg"]["samples_per_s_median"]
                                              / res["finetune_b60"]["store"]["samples_per_s_median"])
    res["finetune_b60"]["steps_per_round"] = steps
    print("finetune", json.dumps(res["finetune_b60"]), flush=True)

    # ---- test_videos: store-fed vs JPEG-fed, same windows and capacity
    model.eval()
    frames = counts[n_train:]
    calls = {"store": lambda: test_videos(model, test_store, frames, labels[n_train:], capacity=60, keep_logits=True),
             "jpeg": lambda: test_videos_jpeg(model, read_test, frames, labels[n_train:], capacity=60, keep_logits=True)}
    out = {k: calls[k]() for k in calls}                 # warm-up, and the results the rates are for
    same = all(torch.equal(out["jpeg"][k], out["store"][k]) for k in ("logits", "predictions")) and \
        out["jpeg"]["hits"] == out["store"]["hits"]
    tv = {k: [] for k in calls}
    for r in range(6):
        for name in (("jpeg", "store") if r % 2 == 0 else ("store", "jpeg")):
            dt, _ = timed(calls[name])
            tv[name].append(n_test / dt)
    res["test_videos"] = {k: {"videos_per_s_median": float(np.median(v)), "per_round": v} for k, v in tv.items()}
    res["test_videos"]["jpeg_over_store"] = (res["test_videos"]["jpeg"]["videos_per_s_median"]
                                             / res["test_videos"]["store"]["videos_per_s_median"])
    res["test_videos"]["clips"] = out["store"]["clips"]
    res["test_videos"]["bit_identical"] = bool(same)
    print("test_videos", json.dumps(res["test_videos"]), flush=True)
    res["gpu_after"] = gpu_state()
    print(json.dumps(res))
    if path:
        with open(path, "w") as f:
            json.dump(res, f, indent=1)
    if not same:
        raise SystemExit("JPEG-fed test_videos differs from the store-fed call")


if __name__ == "__main__":
    main()
