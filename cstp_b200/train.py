"""Epoch-level pretraining driver on the fused step: the loop of main_byol.py:162-269 (`main_worker` / `train_BYOL`)
without its per-step host synchronisation.

What it keeps from the reference:
  * SGD hyper-parameters from `opts` (learning_rate, momentum, weight_decay; main_byol.py:229-232), gradient clipping at 18
    when `opts.clip_grad_norm` (main_byol.py:88-90), `--loss_weight` semantics (main_byol.py:70-73);
  * `CosineAnnealingWarmupRestarts(first_cycle_steps=n_epochs, warmup_steps=0.5*n_epochs, min_lr=1e-5, gamma=0.5)` stepped
    once per epoch (main_byol.py:252-258,269): the first epoch runs at 1e-5;
  * the checkpoint format of main_byol.py:132-140 -- {'epoch': epoch + 1, 'arch', 'state_dict', 'optimizer'} in
    `save_<epoch>.pth`, state-dict keys prefixed with `module.` when the reference would have saved a DDP-wrapped model --
    and the resume rule of :214-215,243-244 (begin epoch parsed from the file name; scheduler state NOT restored, the
    schedule is re-derived from the epoch index);
  * the log columns of main_byol.py:216-225.
What it changes: the six `.item()` host syncs per step (main_byol.py:77-84) become one read-back of the per-step loss
vectors per epoch; the all-reduce of the logged loss (:75) is folded into that read-back.
What it adds on request: per-epoch representation (collapse) statistics of the fused step, and nearest-neighbour
retrieval of the live online network every few epochs (RetrievalMonitor), as extra columns of the epoch's row.
"""
from __future__ import annotations

import os

import torch

from .ops import REPR_STATS
from .scheduler.cosine_anneal import lr_at

LOG_COLUMNS = ["epoch", "loss", "loss_byol", "loss_pred_spa", "loss_pred_tem", "loss_pred_pb", "loss_pred_rot", "acc", "lr"]


def epoch_lr(epoch: int, n_epochs: int, max_lr: float, min_lr: float = 1e-5) -> float:
    """Learning rate of 1-based `epoch` under main_byol.py:252-258 (scheduler.step() runs AFTER each epoch)."""
    return lr_at(epoch - 1, n_epochs, max_lr, min_lr, 0.5 * n_epochs, 1.0, 0.5)


def unwrap(model):
    """The bare R21DBYOL behind the DistributedDataParallel / DataParallel wrapper generate_model may return."""
    return getattr(model, "module", model)


def optimizer_state_dict(model, lr: float = 0.03, momentum: float = 0.9, weight_decay: float = 5e-4,
                         initial_lr: float | None = None, betas=(0.9, 0.999), eps: float = 1e-8) -> dict:
    """torch.optim.SGD state dict of the engine's fused optimiser: momentum buffers addressed by the position of each
    parameter in model.parameters() (frozen target_net entries keep their indices and have no state) and ONE complete
    parameter group -- SGD.load_state_dict replaces the live groups by the saved ones, so every hyper-parameter key of
    torch's SGD has to be there for the reference's `optimizer.load_state_dict(...)` + `optimizer.step()` +
    `CosineAnnealingWarmupRestarts(optimizer, ...)` to work on it (main_byol.py:138,243-258).
    When the engine runs Adam / AdamW, the state dict of torch.optim.Adam / AdamW(lr, betas, eps, weight_decay) instead
    (see _adam_state_dict); `momentum` is then unused."""
    model = unwrap(model)
    eng = model._engine
    if eng.optim_kind != "sgd":
        return _adam_state_dict(model, lr, weight_decay, initial_lr, betas, eps)
    names = [n for n, _ in model.named_parameters()]
    state = {}
    if not eng.first_step:
        for i, n in enumerate(names):
            if n in eng.train.slots:
                state[i] = {"momentum_buffer": eng.train.view(n, eng.mom).detach().clone().cpu()}
    group = {"lr": float(lr), "momentum": float(momentum), "dampening": 0, "weight_decay": float(weight_decay),
             "nesterov": False, "maximize": False, "foreach": None, "differentiable": False, "fused": None,
             "initial_lr": float(lr if initial_lr is None else initial_lr), "params": list(range(len(names)))}
    return {"state": state, "param_groups": [group]}


def _adam_state_dict(model, lr, weight_decay, initial_lr, betas, eps) -> dict:
    """torch.optim.Adam / AdamW state dict of the engine's fused Adam: {"step", "exp_avg", "exp_avg_sq"} per parameter
    that takes part in the update, indexed by position in model.parameters() (target_net and parameters frozen with
    requires_grad = False have no state, as torch gives them none), and ONE parameter group whose keys are those the
    installed torch writes (taken from a throw-away optimiser, so they follow the torch version) plus `initial_lr`."""
    eng = model._engine
    state = {}
    if not eng.first_step:
        for i, (n, p) in enumerate(model.named_parameters()):
            if n in eng.train.slots and p.requires_grad:
                state[i] = {"step": torch.tensor(float(eng.adam_step)),
                            "exp_avg": eng.train.view(n, eng.exp_avg).detach().clone().cpu(),
                            "exp_avg_sq": eng.train.view(n, eng.exp_avg_sq).detach().clone().cpu()}
    cls = torch.optim.AdamW if eng.optim_kind == "adamw" else torch.optim.Adam
    group = cls([torch.zeros(1)], lr=float(lr), betas=tuple(float(b) for b in betas), eps=float(eps),
                weight_decay=float(weight_decay)).state_dict()["param_groups"][0]
    group.update(initial_lr=float(lr if initial_lr is None else initial_lr),
                 params=list(range(sum(1 for _ in model.parameters()))))
    return {"state": state, "param_groups": [group]}


def load_optimizer_state_dict(model, sd: dict, optimizer: str | None = None) -> None:
    """Momentum buffers of an `optim.SGD.state_dict()` (ours or one the reference wrote, main_byol.py:138) -> the
    engine's flat momentum buffer.  Hyper-parameters are not taken from the file: the reference re-creates them from
    `opts` on resume as well (main_byol.py:229-232 builds the optimizer before :243-244 loads the state).
    An `optim.Adam` / `AdamW` state dict (entries with exp_avg / exp_avg_sq / step) restores the engine's Adam moments and
    step count instead.  Whether it continues as "adam" or "adamw" is `optimizer` when given, else the group's
    `decoupled_weight_decay` flag (written by the torch versions that have it), else "adam"."""
    model = unwrap(model)
    eng = model._engine
    if any("exp_avg" in st for st in sd.get("state", {}).values()):
        return _load_adam_state(model, sd, optimizer)
    if optimizer not in (None, "sgd") and any("momentum_buffer" in st for st in sd.get("state", {}).values()):
        raise ValueError(f"an SGD state dict cannot continue as {optimizer}")
    names = [n for n, _ in model.named_parameters()]
    loaded = False
    for i, st in sd.get("state", {}).items():
        buf = st.get("momentum_buffer")
        if buf is not None and names[int(i)] in eng.train.slots:
            eng.train.view(names[int(i)], eng.mom).copy_(buf)
            loaded = True
    eng.first_step = not loaded
    if loaded:
        eng.optim_kind = "sgd"


def _load_adam_state(model, sd: dict, optimizer: str | None) -> None:
    eng = model._engine
    if optimizer is None:
        optimizer = "adamw" if sd["param_groups"][0].get("decoupled_weight_decay") else "adam"
    if optimizer not in ("adam", "adamw"):
        raise ValueError(f"an Adam state dict cannot continue as {optimizer}")
    entries = {int(i): st for i, st in sd["state"].items() if "exp_avg" in st}
    steps = {float(st["step"]) for st in entries.values()}
    if len(steps) != 1:
        raise ValueError(f"the fused Adam step keeps one step count for every parameter; the state dict has {sorted(steps)}")
    eng.first_step = True                        # fresh, zeroed moments of the requested kind, then the file's
    eng.select_optimizer(optimizer)
    names = [n for n, _ in model.named_parameters()]
    for i, st in entries.items():
        if names[i] in eng.train.slots:
            eng.train.view(names[i], eng.exp_avg).copy_(st["exp_avg"])
            eng.train.view(names[i], eng.exp_avg_sq).copy_(st["exp_avg_sq"])
    eng.adam_step = int(steps.pop())
    eng.first_step = False


def save_checkpoint(path: str, model, epoch: int, arch: str, ddp_prefix: bool = True, lr: float = 0.03,
                    momentum: float = 0.9, weight_decay: float = 5e-4, initial_lr: float | None = None,
                    betas=(0.9, 0.999), eps: float = 1e-8) -> None:
    """main_byol.py:132-140.  Keys carry the `module.` prefix of the DDP-wrapped model the reference saves (once: a model
    that is already wrapped contributes it itself).  The optimizer entry is the SGD or Adam / AdamW state dict of
    whichever optimiser the engine runs (optimizer_state_dict)."""
    sd = {}
    for k, v in model.state_dict().items():
        k = k if (k.startswith("module.") or not ddp_prefix) else "module." + k
        sd[k] = v.detach().cpu()
    torch.save({"epoch": epoch + 1, "arch": arch, "state_dict": sd,
                "optimizer": optimizer_state_dict(model, lr, momentum, weight_decay, initial_lr, betas, eps)}, path)


def load_checkpoint(path: str, model, example_clip: torch.Tensor | None = None, optimizer: str | None = None) -> int:
    """Restores weights, BatchNorm buffers and the optimiser state (SGD momentum, or Adam / AdamW moments and step count;
    `optimizer` as in load_optimizer_state_dict); returns the epoch to continue with (the number in the file name,
    main_byol.py:214-215).  `example_clip` (a device tensor of the training shape) binds the engine first so that the
    optimiser buffers have a home."""
    md = torch.load(path, map_location="cpu", weights_only=False)
    sd = {(k[len("module."):] if k.startswith("module.") else k): v for k, v in md["state_dict"].items()}
    model = unwrap(model)
    model.load_state_dict(sd)
    if example_clip is not None:
        model._bind(example_clip)
        load_optimizer_state_dict(model, md["optimizer"], optimizer)
    return int(os.path.basename(path).split("_")[1].split(".")[0])


def pretrain_epochs(model, batches, opts, begin_epoch: int = 1, result_path: str | None = None, arch: str = "r21d_byol-1",
                    grad_sync=None, save_every: int = 100, log=None, optimizer: str = "sgd", betas=(0.9, 0.999),
                    eps: float = 1e-8, collapse_stats: bool = False, monitor: "RetrievalMonitor | None" = None,
                    monitor_every: int = 10):
    """Runs epochs begin_epoch..opts.n_epochs.  `batches(epoch)` yields (clip_1, clip_2, (spa, tem, pb, rot_1, rot_2)) on
    the device.  Returns one dict of LOG_COLUMNS per epoch.  optimizer="adam" / "adamw" (with betas, eps) trains with
    torch.optim.Adam / AdamW semantics; learning rate, weight decay and gradient clipping still come from `opts`.

    collapse_stats=True: every step also computes its representation statistics on the device (R21DBYOL.step_stats);
    their epoch mean comes back with the losses in the same read-back (averaged over ranks like them) and the row gains
    the columns std_feat, std_proj, std_pred, std_tproj and feat_norm, each the mean of the two views.
    monitor (a RetrievalMonitor): every `monitor_every` epochs and at the last epoch, the row gains its recall@k columns,
    computed from the live online network.  Neither changes the training: losses, weights and checkpoints are bit for bit
    those of a run without them."""
    if monitor_every < 1:
        raise ValueError(f"monitor_every must be at least 1, got {monitor_every}")
    rows = []
    wrapped, model = model, unwrap(model)        # the fused step lives on the bare module; checkpoints keep the wrapper's keys
    clip = 18.0 if getattr(opts, "clip_grad_norm", 1) else 0.0
    dist = torch.distributed.is_available() and torch.distributed.is_initialized()
    rank, world = (torch.distributed.get_rank(), torch.distributed.get_world_size()) if dist else (0, 1)
    for epoch in range(begin_epoch, opts.n_epochs + 1):
        lr = epoch_lr(epoch, opts.n_epochs, opts.learning_rate)
        per_step, per_stats = [], []
        for clip_1, clip_2, labels in batches(epoch):
            losses = model.train_step(clip_1, clip_2, labels, opts.loss_weight, lr=lr, momentum=opts.momentum,
                                      weight_decay=opts.weight_decay, clip_grad_norm=clip, grad_sync=grad_sync,
                                      optimizer=optimizer, betas=betas, eps=eps, collapse_stats=collapse_stats)
            per_step.append(losses.clone())                       # device side; no host sync inside the epoch
            if collapse_stats:
                per_stats.append(model.step_stats().clone())
        L = torch.stack(per_step).mean(0)
        if dist:
            torch.distributed.all_reduce(L)                       # reduce_mean of main_byol.py:22-26,75
            L /= world
        if collapse_stats:
            S = torch.stack(per_stats).mean(0)
            if dist:
                torch.distributed.all_reduce(S)
                S /= world
            L, S = torch.cat([L, S.reshape(-1)]).cpu().split([L.numel(), S.numel()])
            S = S.view(per_stats[0].shape)
        else:
            L = L.cpu()
        w = opts.loss_weight
        total = w[0] * L[7] + L[6]
        # main_byol.py:81-84,119-129: pb / rot columns are the MEAN of the two views' terms, acc is None, lr has 5 decimals
        row = dict(zip(LOG_COLUMNS, [epoch, total.item(), L[7].item(), L[0].item(), L[1].item(), ((L[2] + L[3]) / 2).item(),
                                     ((L[4] + L[5]) / 2).item(), None, float("{:.5f}".format(lr))]))
        if collapse_stats:
            row.update({name: ((S[0, i] + S[1, i]) / 2).item() for i, name in enumerate(REPR_STATS)})
        if monitor is not None and (epoch % monitor_every == 0 or epoch == opts.n_epochs):
            row.update(monitor(wrapped, rank, world))
        rows.append(row)
        if log is not None:
            log(row)
        if result_path is not None and (epoch % save_every == 0 or epoch == opts.n_epochs):
            save_checkpoint(os.path.join(result_path, f"save_{epoch}.pth"), wrapped, epoch, arch, lr=lr,
                            momentum=opts.momentum, weight_decay=opts.weight_decay, initial_lr=opts.learning_rate,
                            betas=betas, eps=eps)
    return rows


class RetrievalMonitor:
    """Nearest-neighbour retrieval of the live online network during pretraining (the VCOP / Pace protocol): a call
    extracts per-video features of the gallery (the train split) and of the queries (the test split) from the pretraining
    model itself (evaluate.video_features / video_features_jpeg on R21DBYOL(pretrain=True)), ranks the gallery for every
    query (evaluate.retrieve_videos) and returns {"recall@k": fraction of queries} for every k in `ks`.

    gallery, query: (source, total_frames, labels), source a GpuVideoStore or a read_frames(video, frame_numbers)
    callable returning the JPEG bytes of those frames (frame sizes are read from each video's first frame).  clip_kwargs
    (sample_duration, sample_size, pb_rate, capacity) go to the feature extraction.  The model's training state is left
    as it was, and nothing is written to disk."""

    def __init__(self, gallery, query, ks=(1, 5, 10, 20, 50), **clip_kwargs):
        self.ks = tuple(int(k) for k in ks)
        if not self.ks or min(self.ks) < 1 or max(self.ks) > 64:
            raise ValueError(f"retrieval cutoffs must lie in [1, 64], got {ks}")
        for name, side in (("gallery", gallery), ("query", query)):
            if len(side) != 3 or len(side[1]) != len(side[2]):
                raise ValueError(f"{name}: expected (store or read_frames, total_frames, labels) with one label per video")
        self.gallery, self.query, self.clip_kwargs = tuple(gallery), tuple(query), clip_kwargs

    def _features(self, model, side, rank, world):
        from .data_process.datasets import GpuVideoStore
        from .evaluate import video_features, video_features_jpeg
        source, frames, _ = side
        if isinstance(source, GpuVideoStore):
            return video_features(model, source, frames, rank=rank, world=world, **self.clip_kwargs)
        eng = unwrap(model)._engine
        return video_features_jpeg(model, source, frames, device=eng.device if eng is not None else "cuda", rank=rank,
                                   world=world, **self.clip_kwargs)

    def __call__(self, model, rank: int = 0, world: int = 1) -> dict:
        from .evaluate import retrieve_videos
        g = self._features(model, self.gallery, rank, world)
        q = self._features(model, self.query, rank, world)
        r = retrieve_videos(q, self.query[2], g, self.gallery[2], self.ks, rank=rank, world=world)
        return {f"recall@{k}": r["recall"][k] for k in self.ks}


# ---------------------------------------------------------------------------------------------- finetune driver
class PlateauLR:
    """`optim.lr_scheduler.ReduceLROnPlateau(optimizer, 'min', patience=opts.lr_patience)` of main_ft_mp.py:152 for the
    scalar learning rate of the fused finetune step: mode 'min', factor 0.1, relative threshold 1e-4, no cooldown,
    min_lr 0, eps 1e-8 (torch's defaults), stepped with the epoch's mean validation loss (main_ft_mp.py:292)."""

    def __init__(self, lr: float, patience: int = 10, factor: float = 0.1, threshold: float = 1e-4, eps: float = 1e-8):
        self.lr, self.patience, self.factor, self.threshold, self.eps = float(lr), int(patience), factor, threshold, eps
        self.best = float("inf")
        self.num_bad_epochs = 0

    def step(self, metric: float) -> float:
        metric = float(metric)
        if metric < self.best * (1.0 - self.threshold):
            self.best = metric
            self.num_bad_epochs = 0
        else:
            self.num_bad_epochs += 1
        if self.num_bad_epochs > self.patience:
            new_lr = max(self.lr * self.factor, 0.0)
            if self.lr - new_lr > self.eps:
                self.lr = new_lr
            self.num_bad_epochs = 0
        return self.lr


FT_TRAIN_COLUMNS = ["epoch", "loss", "acc", "lr"]
FT_VAL_COLUMNS = ["epoch", "loss", "acc"]


def finetune_epochs(model, train_batches, val_batches, opts, begin_epoch: int = 1, result_path: str | None = None,
                    arch: str = "r21d_byol-1", grad_sync=None, log_train=None, log_val=None, optimizer: str = "sgd",
                    betas=(0.9, 0.999), eps: float = 1e-8):
    """The epoch loop of main_ft_mp.py:160-170 on the fused finetune step: `train` (:179-244: CrossEntropyLoss, SGD.step,
    top-1 accuracy, mean loss / accuracy per epoch weighted by batch size) then `validation` (:246-310: model.eval(), mean
    loss / accuracy, ReduceLROnPlateau on the validation loss, `save_<epoch>_max.pth` whenever the validation accuracy
    beats the best so far, the previous best file removed).  `train_batches(epoch)` / `val_batches(epoch)` yield
    (clips, labels) on the device.  Losses and hit counts stay on the device inside an epoch (one read-back per phase
    instead of two `.item()`s per step).  optimizer="adam" / "adamw" (with betas, eps) replaces SGD.step by
    Adam / AdamW.step.  Returns (train rows, val rows) with the reference's log columns."""
    model = unwrap(model)
    task = getattr(opts, "task", "ft_all")
    sched = PlateauLR(opts.learning_rate, getattr(opts, "lr_patience", 10))
    best_name, best_acc = next(iter(getattr(opts, "highest_val", {"name": 0}).items()))
    rows_t, rows_v = [], []

    def fold(acc, loss, hits, n):
        w = torch.tensor([float(n)], device=loss.device)
        return (acc[0] + loss.reshape(1) * w, acc[1] + hits.reshape(1).float(), acc[2] + n)

    for epoch in range(begin_epoch, opts.n_epochs + 1):
        model.train()
        acc = None
        for x, labels in train_batches(epoch):
            loss = model.finetune_step(x, labels, lr=sched.lr, momentum=opts.momentum, weight_decay=opts.weight_decay,
                                       grad_sync=grad_sync, optimizer=optimizer, betas=betas, eps=eps)
            eng = model._engine
            hits = (eng.logits[:, :model.num_classes].argmax(1) == labels).sum()          # calculate_accuracy, utils.py:52-65
            z = torch.zeros(1, device=loss.device)
            acc = fold(acc or (z, z.clone(), 0), loss.clone(), hits, x.shape[0])
        if acc is not None:
            s = torch.cat([acc[0], acc[1]])
            if torch.distributed.is_available() and torch.distributed.is_initialized():
                torch.distributed.all_reduce(s[:1])                 # reduce_mean of the loss (main_ft_mp.py:203)
                s[:1] /= torch.distributed.get_world_size()
            s = s.cpu()
            row = dict(zip(FT_TRAIN_COLUMNS, [epoch, s[0].item() / acc[2], s[1].item() / acc[2], float("{:.5f}".format(sched.lr))]))
            rows_t.append(row)
            if log_train is not None:
                log_train(row)
        # ---- validation (main_ft_mp.py:246-310)
        model.eval()
        acc = None
        with torch.no_grad():
            for x, labels in val_batches(epoch):
                model(x, None, o_type=task)                          # eval-mode forward (running statistics)
                eng = model._last_engine                             # an inference engine when x.shape[0] is not the training batch
                eng.cross_entropy(labels)
                hits = (eng.logits[:x.shape[0], :model.num_classes].argmax(1) == labels).sum()
                z = torch.zeros(1, device=eng.loss.device)
                acc = fold(acc or (z, z.clone(), 0), eng.loss.clone(), hits, x.shape[0])
        if acc is None:
            continue
        s = torch.cat([acc[0], acc[1]]).cpu()
        vloss, vacc = s[0].item() / acc[2], s[1].item() / acc[2]
        sched.step(vloss)
        row = dict(zip(FT_VAL_COLUMNS, [epoch, vloss, vacc]))
        rows_v.append(row)
        if log_val is not None:
            log_val(row)
        if vacc > best_acc and result_path is not None:
            old = os.path.join(result_path, best_name)
            if os.path.exists(old):
                os.remove(old)
            best_name, best_acc = f"save_{epoch}_max.pth", vacc
            save_checkpoint(os.path.join(result_path, best_name), model, epoch, arch, lr=sched.lr, momentum=opts.momentum,
                            weight_decay=opts.weight_decay, initial_lr=opts.learning_rate, betas=betas, eps=eps)
        elif vacc > best_acc:
            best_name, best_acc = f"save_{epoch}_max.pth", vacc
    if hasattr(opts, "highest_val"):
        opts.highest_val = {best_name: best_acc}
    return rows_t, rows_v
