"""GPU JPEG decoding (csrc/jpeg_decode.cu) at the sizes of one pretraining batch of 60 samples, next to Pillow on every
host core, and end-to-end pretraining samples/s fed by `JpegPretrainBatches` against `PretrainBatches` on a resident
store of the same frames (alternated in one run).
    python tools/jpeg_bench.py [out.json]

Workloads (4:2:0, quality 90, as frame extraction writes them):
  ucf        1920 frames of 171x128 (60 samples x up to 32 frames), synthetic video content
  ucf_noise  1920 frames of 171x128, uniform noise: the worst case for the serial entropy decode
  kinetics   960 frames of 340x256 (60 samples x 16 distinct frames)
The streams of a batch total well under the 126 MB L2, so repeated decodes read them from L2 after the upload."""
import io
import json
import os
import random
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch
from PIL import Image

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cstp_b200.data_process.datasets import GpuVideoStore, JpegPretrainBatches, PretrainBatches  # noqa: E402
from cstp_b200.data_process.jpeg import GpuJpegDecoder  # noqa: E402
from cstp_b200.synthetic import synthetic_video  # noqa: E402


def encode(img):
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", quality=90, subsampling=2)
    return b.getvalue()


def frames(kind, n, w, h):
    if kind == "noise":
        rng = np.random.default_rng(0)
        return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for _ in range(n)]
    per = 32
    out = []
    for v in range(0, n, per):
        out += list(synthetic_video(min(per, n - v), w, h, v // per))
    return out


def gpu_decode(streams, w, h, reps=20):
    dec = GpuJpegDecoder("cuda")
    outs = list(torch.empty((len(streams), h, w, 3), dtype=torch.uint8, device="cuda"))
    for _ in range(3):
        GpuJpegDecoder.check(dec.decode(streams, [(w, h)] * len(streams), outs))
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        torch.cuda.synchronize()
        a.record()
        dec.decode(streams, [(w, h)] * len(streams), outs)
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(5):
            dec.decode(streams, [(w, h)] * len(streams), outs)
        torch.cuda.synchronize()
    stage = {}
    for e in prof.events():
        for key, name in (("A_entropy", "jpeg_entropy_kernel"), ("B_idct", "jpeg_idct_kernel"),
                          ("C_colour", "jpeg_colour_kernel"), ("upload", "Memcpy HtoD")):
            if name in e.name:
                stage[key] = stage.get(key, 0.0) + e.device_time / 1e3 / 5
    nbytes = sum(len(s) for s in streams)
    med = float(np.median(ms))
    return {"frames": len(streams), "size": [w, h], "bytes_per_frame": nbytes / len(streams),
            "batch_ms_median": med, "batch_ms_min": float(np.min(ms)), "frames_per_s": len(streams) / med * 1e3,
            "MB_per_s": nbytes / med / 1e3, "stage_ms": stage}


def pillow_rate(streams):
    def one(b):
        return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))
    with ThreadPoolExecutor(os.cpu_count()) as ex:
        list(ex.map(one, streams[:64]))
        t0 = time.perf_counter()
        for _ in range(2):
            list(ex.map(one, streams))
        dt = (time.perf_counter() - t0) / 2
    return {"threads": os.cpu_count(), "frames_per_s": len(streams) / dt, "batch_ms": dt * 1e3}


def end_to_end(n_videos=120, n_frames=40, w=171, h=128, batch=60, rounds=4):
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    enc, store = [], GpuVideoStore("cuda")
    for v in range(n_videos):
        vid = synthetic_video(n_frames, w, h, v)
        enc.append([encode(f) for f in vid])
        store.put(v, np.stack([np.asarray(Image.open(io.BytesIO(b)).convert("RGB")) for b in enc[v]]))
    counts = [n_frames] * n_videos

    def read_frames(video, numbers):
        return [enc[video][k - 1] for k in numbers]
    sources = {"jpeg": JpegPretrainBatches(read_frames, counts, batch), "store": PretrainBatches(store, counts, batch)}
    model = R21DBYOL(pretrain=True).cuda()

    def epoch(src, e):
        n = 0
        for x1, x2, labels in src(e):
            model.train_step(x1, x2, labels, (0.1, 1, 1, 1, 1), lr=0.0)
            n += x1.shape[0]
        return n
    random.seed(0)
    np.random.seed(0)
    torch.manual_seed(0)
    for name in sources:                                 # warm-up: engines, graphs, staging buffers
        epoch(sources[name], 0)
    res = {k: [] for k in sources}
    for r in range(rounds):
        for name in (("jpeg", "store") if r % 2 == 0 else ("store", "jpeg")):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = epoch(sources[name], r + 1)
            torch.cuda.synchronize()
            res[name].append(n / (time.perf_counter() - t0))
    out = {k: {"samples_per_s_median": float(np.median(v)), "per_round": v} for k, v in res.items()}
    out["jpeg_over_store"] = out["jpeg"]["samples_per_s_median"] / out["store"]["samples_per_s_median"]
    out["setup"] = {"videos": n_videos, "frames": n_frames, "size": [w, h], "batch": batch,
                    "steps_per_round": n_videos // batch}
    return out


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    res = {"gpu": q[0] if q else None, "host_cores": os.cpu_count(), "workloads": {}}
    for name, kind, n, w, h in (("ucf", "video", 1920, 171, 128), ("ucf_noise", "noise", 1920, 171, 128),
                                ("kinetics", "video", 960, 340, 256)):
        streams = [encode(f) for f in frames(kind, n, w, h)]
        res["workloads"][name] = {"gpu": gpu_decode(streams, w, h), "pillow_all_cores": pillow_rate(streams)}
        print(name, json.dumps(res["workloads"][name]), flush=True)
    res["end_to_end_b60"] = end_to_end()
    print(json.dumps(res))
    if path:
        with open(path, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
