"""Headline benchmark: clips/sec of one `r21d_byol` pretraining step (main_byol.py:60-91) on 16x112x112 clips.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B_per_gpu] [--impl native|reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); per-GPU work is fixed (weak scaling).  Rank 0 prints ONE JSON
line.  A "step" = online fwd (2 views) + predictor + EMA + target fwd (2 views) + BYOL / 6 CE losses + backward +
(grad all-reduce) + clip + SGD + bf16 re-pack, on synthetic U(-1,1) clips and seeded random-init weights.
`value` = samples/s with inputs resident in HBM; `e2e` = the same through R21DBYOL.train_step with pinned HOST clips
and labels copied in and the loss vector copied out every step.  1 clip = 1 sample = two views (SURVEY.md 8d).
`--dump-outputs DIR` writes what the last device-resident timed step left to its caller (rank 0): the loss vector and a
fixed sample of every state_dict entry, as DIR/<name>.npy (see dump_outputs), so two builds can be compared value by value.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOPS_PER_SAMPLE = 339.5e9       # SURVEY.md 8(d): 8F - 2.449 GFLOP (+0.1 heads), F = 42.733 GFLOP per view
LOSS_WEIGHT = (0.1, 1.0, 1.0, 1.0, 1.0)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.path = index, None, None

    def start(self):
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for n, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        os.unlink(self.path)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def workload_config(B: int, world: int, bn: str = "per-GPU (reference semantics)") -> dict:
    """`config` of the JSON line -- identical for the native and the reference arm."""
    return {"workload": f"r21d_byol UCF-101-shaped pretrain step (UcfRepreBYOLSpPre shape), batch {B}/GPU, "
                        "2 views x 3x16x112x112, loss_weight 0.1 1 1 1 1, SGD lr 0.03 m 0.9 wd 5e-4 clip 18",
            "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
            "bn": bn}


def run_reference(args, rank: int):
    """The reference's CPU implementation of the step (its algorithm restated in oracle/cstp_oracle.py -- the Python
    reference itself is not installable and does not travel to the GPU box), all host threads, bounded sample."""
    if rank != 0:
        return
    from oracle import cstp_oracle as O
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from cstp_b200.engine import trainable_param_specs
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Bs = args.ref_batch
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=True)
    state = {k: v.clone() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    trainable = [n for n, _ in trainable_param_specs()]
    x1, x2, labels = O.synthetic_batch(Bs, 0)
    mom: dict = {}
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        O.pretrain_step(state, trainable, x1, x2, labels, list(LOSS_WEIGHT), 0.03, mom)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    v = Bs / sec
    sample = (f"{Bs} full 16x112x112 clips per timed step through the full network -- a bounded sample of the native arm's "
              f"{args.batch}-clip step (BatchNorm over {Bs} instead of {args.batch} samples; the cost per clip is the same)")
    cfg = workload_config(args.batch, args.gpus)
    # the config names the workload both arms are quoted on; what this arm actually ran per step is stated beside it
    cfg.update({"sampled_batch": Bs, "same_config": Bs == args.batch,
                "note": "one CPU process (rank 0) whatever --gpus says: the CPU arm does not scale with the GPU count, so "
                        "ratios against it at N > 1 are not comparable"})
    emit({
        "impl": "reference", "metric": "clips/sec, r21d_byol pretrain step, 16x112x112", "value": v, "unit": "clips/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": v, "unit": "clips/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def cpu_baseline(seconds_budget: float = 25.0) -> dict:
    from oracle import cstp_oracle as O
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from cstp_b200.engine import trainable_param_specs
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    Bs = 2
    torch.manual_seed(1)
    m = R21DBYOL(pretrain=True)
    state = {k: v.clone() for k, v in m.state_dict().items() if not k.endswith("num_batches_tracked")}
    trainable = [n for n, _ in trainable_param_specs()]
    x1, x2, labels = O.synthetic_batch(Bs, 0)
    mom: dict = {}
    t_all, times = time.perf_counter(), []
    while True:
        t0 = time.perf_counter()
        O.pretrain_step(state, trainable, x1, x2, labels, list(LOSS_WEIGHT), 0.03, mom)
        times.append(time.perf_counter() - t0)
        if len(times) >= 2 and (time.perf_counter() - t_all > seconds_budget or len(times) >= 6):
            break
    sec = sum(times[1:]) / len(times[1:])
    return {"value": Bs / sec, "unit": "clips/s", "cores": cores, "kind": "port",
            "sample": f"oracle/cstp_oracle.pretrain_step on {Bs} full 16x112x112 clips, {len(times) - 1} timed steps after 1 warm-up"}


def config5_record(args, rank: int, world: int) -> dict | None:
    """BASELINE config 5 (Kinetics-400 recipe, README.md:41-49): GLOBAL batch 128 split contiguous-by-rank (utils.py:111),
    BatchNorm statistics over every rank (north-star SyncBN; row exchange over NVLink peer memory), NT-Xent over the
    all-gathered projector outputs of both views (global negatives, loss/NTXent.py with batch_size = the global batch,
    main_byol.py:191-196), gradient all-reduce.  Timed like the main arm; beside it (a) the same build's one-GPU step at
    the same per-GPU batch without any cross-rank exchange -- the denominator of a scaling efficiency -- and (b) the first
    step from the seeded init compared with ONE GPU stepping the whole global batch (N x 128/N == 1 x 128)."""
    import gc
    import torch.distributed as dist
    from cstp_b200 import parallel
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from cstp_b200.synthetic import synthetic_batch
    GB = 128
    b = parallel.per_rank_batch(GB, world)
    lo, hi = parallel.shard_bounds(GB, rank, world)
    gx1, gx2, glab = synthetic_batch(GB, seed=0)
    x1, x2 = gx1[lo:hi].contiguous().cuda(), gx2[lo:hi].contiguous().cuda()
    lab = tuple(l[lo:hi].contiguous().cuda() for l in glab)
    nx = {"weight": 1.0, "temperature": 0.1}
    sync = parallel.GradSync()
    try:
        bn, bn_name = parallel.BnSyncP2P(), "world-p2p (one peer-memory exchange kernel per BatchNorm call)"
    except Exception as e:  # noqa: BLE001   symmetric memory unavailable: the NCCL all-reduce path
        bn, bn_name = parallel.BnSync(), f"world-nccl (all-reduce per BatchNorm call; peer-memory path unavailable: {e})"

    def make(opts):
        torch.manual_seed(1)
        m = R21DBYOL(pretrain=True).cuda()
        m.engine_options = opts
        return m

    def step(m, a, c, lb, gs):
        return m.train_step(a, c, lb, LOSS_WEIGHT, lr=0.09, momentum=0.9, weight_decay=5e-4, clip_grad_norm=18.0, grad_sync=gs)

    def timed(m, gs):
        for _ in range(max(args.warmup, 3)):
            step(m, x1, x2, lab, gs)
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step(m, x1, x2, lab, gs)
        e1.record()
        dist.barrier()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / args.steps

    # ---- data parallel, world statistics, gathered NT-Xent
    dp = make({"bn_sync": bn, "ntxent": {**nx, "gather": True}})
    first = step(dp, x1, x2, lab, sync).clone()
    first_nx = dp._engine.ntxent_loss.clone()
    mean_first = first.clone()
    dist.all_reduce(mean_first)
    mean_first /= world
    ms_dp = timed(dp, sync)
    if hasattr(bn, "check"):
        bn.check()                        # a timed-out peer exchange must not produce a number
    del dp
    gc.collect()
    torch.cuda.empty_cache()
    # ---- denominator: the same per-GPU batch on one GPU, nothing exchanged
    local = make({"ntxent": dict(nx)})
    ms_local = timed(local, None)
    del local
    gc.collect()
    torch.cuda.empty_cache()
    # ---- parity: one GPU steps the whole global batch once
    parity = None
    if rank == 0:
        try:                          # (rank 0 alone: a failure here must not desynchronise the barrier below)
            whole = make({"ntxent": dict(nx)})
            w = step(whole, gx1.cuda(), gx2.cuda(), tuple(l.cuda() for l in glab), None).cpu()
            wnx = whole._engine.ntxent_loss.item()
            mf = mean_first.cpu()
            tot = lambda v, n: LOSS_WEIGHT[0] * v[7].item() + v[6].item() + nx["weight"] * n     # noqa: E731
            parity = {"what": f"first step from the seeded init: {world} ranks x {b} samples vs ONE GPU x {GB} samples "
                              "(same clips, labels and weights)",
                      "loss_total_dp": tot(mf, first_nx.item()), "loss_total_one_gpu": tot(w, wnx),
                      "loss_total_rel": abs(tot(mf, first_nx.item()) - tot(w, wnx)) / abs(tot(w, wnx)),
                      "loss_byol_dp": mf[7].item(), "loss_byol_one_gpu": w[7].item(),
                      "ntxent_dp": first_nx.item(), "ntxent_one_gpu": wnx,
                      "ce_rel_max": max(abs(mf[i].item() - w[i].item()) / abs(w[i].item()) for i in range(6))}
            del whole
        except Exception as e:  # noqa: BLE001
            parity = {"error": f"{type(e).__name__}: {e}"}
        gc.collect()
        torch.cuda.empty_cache()
    dist.barrier()
    if rank != 0:
        return None
    return {"workload": "r21d_byol Kinetics-400-shaped pretrain step (Kin400RepreLMDB shape), GLOBAL batch 128, 2 views x "
                        "3x16x112x112, SyncBN over all ranks + NT-Xent (tau 0.1, weight 1) on the all-gathered projector "
                        "outputs, SGD lr 0.09 m 0.9 wd 5e-4 clip 18",
            "global_batch": GB, "per_gpu_batch": b, "parallelism": f"dp{world}", "scaling": "strong", "bn_sync": bn_name,
            "ntxent": {"rows": 2 * GB, "d": 512, "gather": "all_gather of 2 x (per_gpu_batch, 512) per step"},
            "ms_per_step": ms_dp, "value": GB / (ms_dp * 1e-3), "unit": "clips/s",
            "denominator": {"what": "same build, ONE GPU, the same per-GPU batch, per-GPU BatchNorm, local NT-Xent, no collective "
                                    "(max over ranks); N x its rate is the ceiling of this configuration",
                            "ms_per_step": ms_local, "clips_per_s_times_n": world * b / (ms_local * 1e-3)},
            "parity": parity}


_JSON_OUT = None


def claim_stdout():
    """The driver reads ONE JSON line from stdout.  Libraries print there too (NCCL's version banner under NCCL_DEBUG), so
    file descriptor 1 is pointed at stderr for the rest of the process and the JSON line goes to a private duplicate of the
    original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    claim_stdout()
    _JSON_OUT.write(json.dumps(line) + "\n")
    _JSON_OUT.flush()


def run_with_watchdog(seconds: float, fn, on_timeout):
    """fn() under a watchdog THREAD (the main thread may sit in a CUDA or NCCL call that never returns, where a signal
    handler would not run): on_timeout() is called from the timer thread if fn has not returned after `seconds`."""
    import threading
    dog = threading.Timer(seconds, on_timeout)
    dog.daemon = True
    dog.start()
    try:
        return fn()
    finally:
        dog.cancel()


def bail_out(line: dict | None, key: str, message: str) -> None:
    """Ends the process with exit code 0 from a watchdog: the rank that holds the measured line prints it with the error
    recorded under `key` first (the other ranks pass None)."""
    if line is not None:
        line[key] = {"error": message}
        emit(line)
    sys.stdout.flush()
    os._exit(0)


def ncu_traffic(kernel: str, B: int):
    """(bytes, source): average DRAM bytes (read + write) per launch of `kernel` from the newest committed ncu capture of
    this command at the same per-GPU batch (profiles/rNN_ncu_<kernel>_b<B>_dram.csv: dram__bytes_read.sum +
    dram__bytes_write.sum per launch), or (None, None).  The number is NOT measured in this run: `source` names the file
    so that a reader can check it against the kernel revision."""
    import csv
    import glob
    pat = os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles",
                       "r[0-9][0-9]_ncu_%s_b%d_dram.csv" % (kernel.replace("_kernel", ""), B))
    paths = sorted(glob.glob(pat))
    if not paths:
        return None, None
    total, ids = 0.0, set()
    with open(paths[-1]) as f:
        head = f.readline()
        if head.startswith("#"):          # provenance line of the capture (commit, command)
            note = head[1:].strip()
        else:
            note = None
            f.seek(0)
        for r in csv.reader(f):
            if len(r) > 10 and r[0].isdigit() and r[-3].startswith("dram__bytes_"):
                total += float(r[-1].replace(",", ""))
                ids.add(r[0])
    src = os.path.relpath(paths[-1], os.path.dirname(os.path.abspath(__file__)))
    return (total / len(ids) if ids else None), (src + (" [" + note + "]" if note else ""))


DUMP_SAMPLE = 16384             # values kept of a larger tensor: r21d_byol's 351 state entries come to 4.1 MB
DUMP_LIMIT = 64 << 20


def dump_sample(t: torch.Tensor, k: int = DUMP_SAMPLE) -> torch.Tensor:
    """t flattened; above k elements, the values at k seeded positions that depend only on t's size (the same on every run)."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= k:
        return flat
    idx = torch.randint(0, flat.numel(), (k,), generator=torch.Generator().manual_seed(0))
    return flat[idx.to(flat.device)]


def dump_outputs(out_dir: str, losses: torch.Tensor, state: dict) -> int:
    """Writes what one train_step hands its caller -- the returned loss vector and the module state it leaves -- as
    <out_dir>/losses.npy (the 8 values of R21DBYOL.train_step) and <out_dir>/state.<key>.npy per state_dict entry
    (dump_sample of it).  Floating-point values as float32, integer counters as float64.  Returns the bytes written."""
    import numpy as np
    arrays = {"losses": losses, **{f"state.{k}": dump_sample(v) for k, v in state.items()}}
    arrays = {n: t.detach().cpu().numpy().astype(np.float32 if t.is_floating_point() else np.float64)
              for n, t in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise ValueError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT}-byte budget")
    os.makedirs(out_dir, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=60, help="samples per GPU (UcfRepreBYOLSpPre config: 60)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--ref-batch", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-config5", action="store_true", help="N > 1: skip the BASELINE config 5 sub-record")
    ap.add_argument("--config5-timeout", type=float, default=240.0, help="seconds before a hung config 5 sub-record is cut off")
    ap.add_argument("--bn-sync", default="local", choices=["local", "world", "world-p2p"],
                    help="local: per-GPU BatchNorm statistics (the reference's behaviour); world: SyncBN over all ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss vector and a fixed sample of the model state after the last timed step as "
                         "DIR/<name>.npy (rank 0).  Native arm only: the reference arm times a sampled batch of "
                         "--ref-batch clips, not the --batch clips of the native step, so its outputs would not compare")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the native arm's outputs")
    claim_stdout()
    from cstp_b200 import parallel
    rank, world, local = parallel.env_world()
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not parallel.wait_for_cuda() or not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the native path has no CPU fallback (use --impl reference for the CPU arm)")
    warm = max(args.warmup, 3)
    torch.cuda.set_device(local)
    # NCCL's own banner / debug lines (NCCL_DEBUG may be set by the environment) must not land on stdout: one JSON line only
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    parallel.init_from_env("nccl")
    import torch.distributed as dist
    from cstp_b200 import ops
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from cstp_b200.synthetic import synthetic_batch   # seeded input protocol (SURVEY.md 8d)

    B = args.batch
    torch.manual_seed(1)
    model = R21DBYOL(pretrain=True).cuda()
    if args.bn_sync == "world" and world > 1:
        model.engine_options = {"bn_sync": parallel.BnSync()}
    elif args.bn_sync == "world-p2p" and world > 1:
        model.engine_options = {"bn_sync": parallel.BnSyncP2P()}
    hx1, hx2, hlabels = synthetic_batch(B, seed=rank)
    hx1, hx2 = hx1.pin_memory(), hx2.pin_memory()
    hlabels = tuple(l.pin_memory() for l in hlabels)
    x1, x2 = hx1.cuda(), hx2.cuda()
    labels = tuple(l.cuda() for l in hlabels)
    sync = parallel.GradSync() if world > 1 else None

    def step(a, b, lab):
        return model.train_step(a, b, lab, LOSS_WEIGHT, lr=0.03, momentum=0.9, weight_decay=5e-4, clip_grad_norm=18.0,
                                grad_sync=sync)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warm):
        step(x1, x2, labels)
    barrier()

    # ---------------- device-resident timed region
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = ops.launch_count()
    barrier()
    e0.record()
    for _ in range(args.steps):
        losses = step(x1, x2, labels)
    e1.record()
    barrier()
    launches = ops.launch_count() - l0
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_step = ms.item() / args.steps
    bs = getattr(model, "engine_options", {}).get("bn_sync")
    if hasattr(bs, "check"):
        bs.check()                        # a timed-out peer exchange must not produce a number
    clk = clocks.stop() if rank == 0 else None
    final = losses.tolist()
    if args.dump_outputs and rank == 0:
        # before the end-to-end region steps the same model on: `losses` and the state are the last timed step's
        dump_outputs(args.dump_outputs, losses, model.state_dict())

    # ---------------- end-to-end region: pinned host clips in, loss vector out, every step.  Each step's clips and labels
    # are copied host -> device inside the timed region (the copy of step i+1 runs on a side stream while step i
    # computes, as the reference's data_prefetcher does), and every step's loss vector is copied into pinned host memory
    # behind that step and consumed by the host (cstp_b200.data.LossReadback: the host collects a vector a few steps after it
    # was produced instead of stalling the launch thread on it; all of them are collected before the region ends).
    from cstp_b200.data import ClipPrefetcher, LossReadback
    rb = LossReadback(8)
    barrier()
    e0.record()
    pf = ClipPrefetcher(((hx1, hx2, hlabels) for _ in range(args.steps)))
    while True:
        batch = pf.next()
        if batch is None:
            break
        out = step(*batch)
        pf.done()
        rb.push(out)
    host_losses = rb.drain()
    assert len(host_losses) == args.steps and all(v == v for row in host_losses for v in row)      # every step read, no NaN
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    if world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms_e2e = ms2.item() / args.steps
    h2d = pf.h2d_bytes

    # ---------------- roofline of the dominant kernel family (tcgen05 implicit-GEMM conv: fwd + dgrad launches)
    pk = peaks()
    roof = None
    # the instrumented step runs on EVERY rank (with world-synchronised BatchNorm it contains collectives); rank 0 reports
    model._engine.profile_tensor_launches(x1, x2)
    if rank == 0:
        eng = model._engine
        kern: dict = {}
        for kind, tag, t_ms, fl, n, name in eng.last_profile:
            k = kern.setdefault(name, {"ms_per_step": 0.0, "flops": 0.0, "launches_per_step": 0})
            k["ms_per_step"] += t_ms
            k["flops"] += fl
            k["launches_per_step"] += n
        for k in kern.values():
            k["tflops"] = k["flops"] / (k["ms_per_step"] * 1e-3) / 1e12 if k["ms_per_step"] > 0 else 0.0
            k["share_of_step"] = k["ms_per_step"] / ms_step
            k["avg_launch_ms"] = k["ms_per_step"] / max(1, k["launches_per_step"])
            del k["flops"]
        dom = max(kern, key=lambda k: kern[k]["ms_per_step"])
        ach = kern[dom]["tflops"]
        # the dominant kernel's launches by layer family: its average mixes tensor-bound launches (64 -> 144 1x3x3) with
        # launches that are HBM-bound by their operands (3x1x1 on 144-channel tensors, the 3- / 45-channel stem) or carry
        # the BatchNorm + ReLU operand prologue of the pass they replace
        fam: dict = {}
        for kind, tag, t_ms, fl, n, name in eng.last_profile:
            if name != dom:
                continue
            layer = tag.split(".", 1)[1] if "." in tag else tag
            group = kind + (" stem" if layer.startswith("conv1.") else " 1x3x3" if layer.endswith("spatial") else " 3x1x1")
            f = fam.setdefault(group, {"ms_per_step": 0.0, "flops": 0.0, "launches_per_step": 0})
            f["ms_per_step"] += t_ms
            f["flops"] += fl
            f["launches_per_step"] += n
        for f in fam.values():
            f["tflops"] = f["flops"] / (f["ms_per_step"] * 1e-3) / 1e12 if f["ms_per_step"] > 0 else 0.0
            f["frac_of_peak"] = f["tflops"] / pk["tf_sustained"]
            del f["flops"]
        tensor_ms = sum(k["ms_per_step"] for k in kern.values())
        traffic, traffic_src = ncu_traffic(dom, B)
        roof = {"bound": "tensor", "kernel": dom, "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                "frac": ach / pk["tf_sustained"], "traffic": traffic, "traffic_source": traffic_src,
                "traffic_how": "bytes per launch: dram__bytes_read.sum + dram__bytes_write.sum averaged over the kernel's launches "
                               "of one step in a COMMITTED ncu capture of this command (traffic_source; not measured in this "
                               "run; null: no capture at this batch)",
                "peak_source": pk["src"] + " sustained bf16 cuBLAS matmul (kernel timed inside a long step)",
                "how": "CUDA events on the launching stream around every launch of the kernel in one extra instrumented "
                       "step; achieved = sum over its launches of 2*M*N*K (true channel counts) / sum of durations",
                "kernels": kern, "dominant_by_layer_family": fam,
                "all_tensor_kernels_tflops": B * FLOPS_PER_SAMPLE / (tensor_ms * 1e-3) / 1e12,
                "step_tflops": B * FLOPS_PER_SAMPLE / (ms_step * 1e-3) / 1e12}
    value = world * B / (ms_step * 1e-3)
    line = None
    if rank == 0:
        line = {
            "metric": "clips/sec, r21d_byol pretrain step, 16x112x112", "value": value, "unit": "clips/s", "n_gpus": world,
            "steps": args.steps, "warmup": warm, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {**workload_config(B, world, "per-GPU (reference semantics)" if args.bn_sync == "local" or world == 1
                                         else ("world-synchronised (SyncBN all-reduce per BatchNorm call)" if args.bn_sync == "world" else
                                               "world-synchronised (SyncBN rows exchanged over NVLink peer memory, one kernel per call)")),
                       "l2_policy": "inputs and activations far larger than the 126 MB L2 (clips alone 2x%.0f MB)" % (x1.numel() * 4 / 1e6),
                       "views_per_s": 2 * value, "schedule": "two streams (target fwd || online fwd, wgrad || BN backward)"},
            "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "clips/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 32,
                    "ms_per_step": ms_e2e},
            "gpu_launches": int(launches), "clocks": clk, "roofline": roof, "cpu_baseline": None,
            "losses_last_step": {"byol": final[7], "ce": final[:6]},
        }
    c5 = None
    if world > 1 and not args.no_config5:
        eng = None                        # (rank 0's handle from the roofline block) the batch-60 engine must go first
        del model
        import gc
        gc.collect()
        torch.cuda.empty_cache()

        # the batch-60 line above is already measured: a sub-record that raises is reported, one that HANGS (a lost peer in
        # an exchange) is cut off by a watchdog thread on every rank -- rank 0 prints the line with the error, all exit 0
        def sub_record():
            try:
                c = config5_record(args, rank, world)
            except Exception as e:  # noqa: BLE001
                import traceback
                traceback.print_exc()
                c = {"error": f"{type(e).__name__}: {e}"} if rank == 0 else None
            dist.barrier()
            return c
        c5 = run_with_watchdog(args.config5_timeout, sub_record, lambda: bail_out(
            line, "config5", f"config-5 sub-record did not finish within {args.config5_timeout} s"))
    elif world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline()
    if c5 is not None:
        line["config5"] = c5
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
