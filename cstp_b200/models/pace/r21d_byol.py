"""Drop-in `r21d_byol` module family backed by the B200 step engine.

Mirrors the public surface of the reference's models/pace/r21d_byol.py -- class names, constructor arguments,
sub-module / parameter / buffer names and registration order (checkpoints are keyed by them, SURVEY.md A.5), the
glorot re-initialisation (:301-329) and `forward(x1, x2, o_type)` (:357-401) -- but none of the sub-modules computes
anything: they only hold parameters.  All arithmetic of `o_type="loss_com"` runs in cstp_b200.engine.StepEngine
(hand-written sm_100a kernels behind the C ABI); the nn.Parameters are re-pointed at the engine's flat fp32 buffers
on first use, so `state_dict()`, `load_state_dict()`, `optimizer.step()` and DDP all see the live weights.

Two ways to run a step:
  * drop-in:  loss, preds = model(x1, x2, o_type="loss_com"); (...CrossEntropyLoss...).backward(); optimizer.step()
              -- the unmodified loop body of main_byol.py:60-91 works (autograd sees one custom Function);
  * fused:    model.train_step(x1, x2, labels, loss_weight, lr, ...) -- losses, backward, (all-reduce), clip + SGD
              and the bf16 re-pack as one launch program without host synchronisation.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from ... import engine as _engine_mod


def get_fine_tuning_parameters(model, ft_begin_index):
    """Same contract as r21d_byol.py:10-35 (including its quirk: stages are named conv1..conv5, so any
    1 <= ft_begin_index <= 4 selects only `classify`, SURVEY.md A.5)."""
    if ft_begin_index == 0:
        return model.parameters()
    wanted = [f"layer{i}" for i in range(ft_begin_index, 5)] if ft_begin_index <= 4 else []
    wanted.append("classify")
    groups = []
    for name, p in model.named_parameters():
        if any(w in name for w in wanted):
            groups.append({"params": p})
        else:
            p.requires_grad = False
            groups.append({"params": p, "lr": 0.0})
    return groups


class _Holder(nn.Module):
    """Parameter container: the engine computes, sub-modules are never called on their own."""

    def forward(self, *a, **k):
        raise RuntimeError(f"{type(self).__name__} only holds parameters; call R21DBYOL.forward / train_step "
                           "(the computation runs in the cstp_b200 CUDA engine, there is no per-module path)")


def _triple(v):
    return tuple(v) if isinstance(v, (tuple, list)) else (v, v, v)


class SpatioTemporalConv(_Holder):
    """(1,kH,kW) spatial conv -> BatchNorm3d -> ReLU -> (kT,1,1) temporal conv; parameters of r21d_byol.py:52-92."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, bias=False, first_conv=False):
        super().__init__()
        k, s, p = _triple(kernel_size), _triple(stride), _triple(padding)
        mid = _engine_mod.intermed_channels(in_channels, out_channels, k)
        self.spatial_conv = nn.Conv3d(in_channels, mid, (1, k[1], k[2]), stride=(1, s[1], s[2]),
                                      padding=(0, p[1], p[2]), bias=bias)
        self.bn = nn.BatchNorm3d(mid)
        self.temporal_conv = nn.Conv3d(mid, out_channels, (k[0], 1, 1), stride=(s[0], 1, 1), padding=(p[0], 0, 0),
                                       bias=bias)


class SpatioTemporalResBlock(_Holder):
    """Parameters of r21d_byol.py:113-139 (downsample members are registered first)."""

    def __init__(self, in_channels, out_channels, kernel_size, downsample=False):
        super().__init__()
        self.downsample = downsample
        pad = kernel_size // 2
        if downsample:
            self.downsampleconv = SpatioTemporalConv(in_channels, out_channels, 1, stride=2)
            self.downsamplebn = nn.BatchNorm3d(out_channels)
        self.conv1 = SpatioTemporalConv(in_channels, out_channels, kernel_size, padding=pad,
                                        stride=2 if downsample else 1)
        self.bn1 = nn.BatchNorm3d(out_channels)
        self.conv2 = SpatioTemporalConv(out_channels, out_channels, kernel_size, padding=pad)
        self.bn2 = nn.BatchNorm3d(out_channels)


class SpatioTemporalResLayer(_Holder):
    def __init__(self, in_channels, out_channels, kernel_size, layer_size, block_type=SpatioTemporalResBlock,
                 downsample=False):
        super().__init__()
        if layer_size != 1:
            raise ValueError("the B200 engine implements the (1,1,1,1) layout R21DBYOL uses (r21d_byol.py:268)")
        self.block1 = block_type(in_channels, out_channels, kernel_size, downsample)
        self.blocks = nn.ModuleList([])


def _mlp(cin, hidden, cout):
    return nn.Sequential(nn.Linear(cin, hidden), nn.BatchNorm1d(hidden), nn.ReLU(inplace=True), nn.Linear(hidden, cout))


class Projector(_Holder):
    def __init__(self, dim, projection_size, projection_hidden_size=4096):
        super().__init__()
        self.net = _mlp(dim, projection_hidden_size, projection_size)


class Predictor(_Holder):
    def __init__(self, dim, prediction_size, prediction_hidden_size=4096):
        super().__init__()
        self.net = _mlp(dim, prediction_hidden_size, prediction_size)


class R2Plus1DNet(_Holder):
    def __init__(self, layer_sizes=(1, 1, 1, 1), block_type=SpatioTemporalResBlock, proj_flag=False):
        super().__init__()
        self.conv1 = SpatioTemporalConv(3, 64, (3, 7, 7), stride=(1, 2, 2), padding=(1, 3, 3))
        self.bn1 = nn.BatchNorm3d(64)
        self.conv2 = SpatioTemporalResLayer(64, 64, 3, layer_sizes[0], block_type=block_type)
        self.conv3 = SpatioTemporalResLayer(64, 128, 3, layer_sizes[1], block_type=block_type, downsample=True)
        self.conv4 = SpatioTemporalResLayer(128, 256, 3, layer_sizes[2], block_type=block_type, downsample=True)
        self.conv5 = SpatioTemporalResLayer(256, 512, 3, layer_sizes[3], block_type=block_type, downsample=True)
        self.proj_flag = proj_flag
        if proj_flag:
            self.project = Projector(dim=512, projection_size=512, projection_hidden_size=4096)


class _LossComFn(torch.autograd.Function):
    """One autograd node for the whole `loss_com` forward; backward runs the engine's backward program."""

    @staticmethod
    def forward(ctx, model, x1, x2, *params):
        eng = model._engine
        eng.forward(x1, x2, repack_online=True)
        ctx.model = model
        outs = [eng.losses[7].clone()] + [t[:, :5].clone() for t in eng.logits6]
        return tuple(outs)

    @staticmethod
    def backward(ctx, g_loss, *g_logits):
        model = ctx.model
        eng = model._engine
        if g_loss is None:
            eng.byol_scale.zero_()
        else:
            eng.byol_scale.copy_(g_loss.reshape(1))
        for buf, g in zip(eng.dlogits6, g_logits):
            buf.zero_()
            if g is not None:
                buf[:, :5].copy_(g)
        eng.backward()
        grads = [eng.train.view(n, eng.grad).clone() for n in model._trainable_names]
        return (None, None, None, *grads)


class _FinetuneFn(torch.autograd.Function):
    """One autograd node for the finetune forward (backbone + normalise + cls_bn + classify)."""

    @staticmethod
    def forward(ctx, model, x, *params):
        eng = model._engine
        eng.eval_mode = False
        eng.forward(x, repack=True)
        ctx.model = model
        return eng.logits[:, :model.num_classes].clone()

    @staticmethod
    def backward(ctx, g):
        model = ctx.model
        eng = model._engine
        eng.dlogits.zero_()
        eng.dlogits[:, :model.num_classes].copy_(g)
        eng.backward()
        grads = [eng.train.view(n, eng.grad).clone() for n in model._trainable_names]
        return (None, None, *grads)


class R21DBYOL(nn.Module):
    """Drop-in for r21d_byol.py:260-401: pretrain=True is the `loss_com` pretraining model, pretrain=False the
    finetune / test model (`ft_fc`, `ft_all`, `test`) with `num_classes` and `cls_bn` keyword arguments."""

    def __init__(self, pretrain=True, momentum=0.996, **kwargs):
        super().__init__()
        self.pretrain = bool(pretrain)
        if pretrain:
            self.momentum = momentum
            self.online_net = R2Plus1DNet(layer_sizes=(1, 1, 1, 1), proj_flag=True)
            self.target_net = R2Plus1DNet(layer_sizes=(1, 1, 1, 1), proj_flag=True)
            self.predictor = Predictor(dim=512, prediction_size=512, prediction_hidden_size=4096)
            for p in self.target_net.parameters():
                p.requires_grad = False
            self.overlap_spa = _mlp(1024, 1024, 5)
            self.overlap_tem = _mlp(1024, 1024, 5)
            self.pb_cls = _mlp(512, 512, 5)
            self.rotate_cls = _mlp(512, 512, 5)
        else:
            self.online_net = R2Plus1DNet(layer_sizes=(1, 1, 1, 1), proj_flag=False)
            self.num_classes = kwargs["num_classes"]
            self.classify = nn.Linear(512, self.num_classes)
            self.cls_bn = kwargs["cls_bn"]
            if self.cls_bn:
                self.cls_bn = nn.BatchNorm1d(512)
        # r21d_byol.py:301-329: every Linear / Conv3d / BatchNorm weight (BN gamma included) is redrawn
        # U(+-sqrt(6/(fan_in+fan_out))); 1-D tensors use fan_in = fan_out = C/2.
        with torch.no_grad():
            for m in self.modules():
                if isinstance(m, (nn.Linear, nn.Conv3d, nn.BatchNorm1d, nn.BatchNorm3d)):
                    w = m.weight
                    if w.dim() < 2:
                        fan_in = fan_out = int(w.size(0) / 2)
                    else:
                        rf = w[0][0].numel() if w.dim() > 2 else 1
                        fan_in, fan_out = w.size(1) * rf, w.size(0) * rf
                    bound = math.sqrt(6.0 / float(fan_in + fan_out))
                    w.uniform_(-bound, bound)
        self._engine = None
        self._engine_key = None
        self._infer = {}              # (capacity, T, H, W, device) -> engine_ft.InferenceEngine (eval forwards)
        self._infer_owner = None      # the inference engine that owns the stores while no engine is bound
        self._last_engine = None      # the engine that ran the last forward
        self._wgen = 0                # weight generation (see _repack_if_changed)
        if pretrain:
            self._trainable_names = [n for n, _ in _engine_mod.trainable_param_specs()]
        else:
            from ... import engine_ft
            self._trainable_names = [n for n, _ in engine_ft.finetune_param_specs(self.num_classes, bool(self.cls_bn))]
        self._dirty = True

    # ------------------------------------------------------------------------------------------ engine binding
    def _bind(self, x1):
        """Creates (or re-binds after .cuda()/.to()) the step engine for this batch geometry and aliases every
        parameter / BN buffer of the module tree onto the engine's flat buffers."""
        _engine_mod.ops.require_device(x1)
        B, _, T, H, W = x1.shape
        key = (B, T, H, W, x1.device)
        eng = self._engine
        if eng is None or self._engine_key != key:
            new = _engine_mod.StepEngine(B, T, H, W, device=x1.device, momentum_ema=self.momentum,
                                         **getattr(self, "engine_options", {}))
            if eng is not None:      # keep optimiser-side state across a batch-geometry change
                new.take_optimizer_state(eng)
            self._infer.clear()      # feature engines read the stores of the engine being replaced
            eng = self._engine = new
            self._engine_key = key
            self._alias_ptr = None
        sentinel = self.online_net.conv1.spatial_conv.weight
        if self._alias_ptr != sentinel.data_ptr():
            with torch.no_grad():
                for name, p in self.named_parameters():
                    store = eng.target if name.startswith("target_net.") else eng.train
                    v = store.view(name)
                    v.copy_(p.data)
                    p.data = v
                nbt, inc = [], []
                for mname, mod in self.named_modules():
                    if isinstance(mod, (nn.BatchNorm1d, nn.BatchNorm3d)):
                        for b in ("running_mean", "running_var"):
                            v = eng.bufs.view(f"{mname}.{b}")
                            v.copy_(mod._buffers[b])
                            mod._buffers[b] = v
                        nbt.append(mod)
                        inc.append(1 if mname in ("overlap_spa.1", "overlap_tem.1") else 2)
                flat = torch.stack([m._buffers["num_batches_tracked"].to(x1.device) for m in nbt])
                for i, m in enumerate(nbt):
                    m._buffers["num_batches_tracked"] = flat[i]
                self._nbt, self._nbt_inc = flat, torch.tensor(inc, device=x1.device, dtype=flat.dtype)
            eng.drop_graph()                     # a captured step holds the old num_batches_tracked tensors
            self._alias_ptr = sentinel.data_ptr()
            self._dirty = True
        return eng

    def _ft_key(self, x):
        B, _, T, H, W = x.shape
        bgrads = any(p.requires_grad for n, p in self.named_parameters() if n.startswith("online_net."))
        return (B, T, H, W, x.device, bgrads)

    def _bind_ft(self, x):
        """Finetune / test flavour of _bind: a FinetuneEngine per (batch geometry, frozen-backbone) configuration."""
        from ... import engine_ft
        _engine_mod.ops.require_device(x)
        if not isinstance(self.cls_bn, nn.Module):
            raise TypeError("'bool' object is not callable")      # the reference calls self.cls_bn(feat) unconditionally
        B, _, T, H, W = x.shape
        key = self._ft_key(x)
        eng = self._engine
        if eng is None or self._engine_key != key:
            new = engine_ft.FinetuneEngine(B, T, H, W, device=x.device, num_classes=self.num_classes, cls_bn=True,
                                           backbone_grads=key[-1], **getattr(self, "engine_options", {}))
            if eng is not None:
                new.take_optimizer_state(eng)
            self.free_inference_engines()        # they read the stores the parameters are about to leave
            eng = self._engine = new
            self._engine_key = key
            self._alias_ptr = None
        self._alias_ft(eng)
        return eng

    def _alias_ft(self, eng):
        """Points every parameter / BatchNorm buffer at eng's flat stores (again after .cuda() / .to() moved them)."""
        sentinel = self.online_net.conv1.spatial_conv.weight
        if getattr(self, "_alias_ptr", None) != sentinel.data_ptr():
            with torch.no_grad():
                for name, p in self.named_parameters():
                    v = eng.train.view(name)
                    v.copy_(p.data)
                    p.data = v
                nbt = []
                for mname, mod in self.named_modules():
                    if isinstance(mod, (nn.BatchNorm1d, nn.BatchNorm3d)):
                        for b in ("running_mean", "running_var"):
                            v = eng.bufs.view(f"{mname}.{b}")
                            v.copy_(mod._buffers[b])
                            mod._buffers[b] = v
                        nbt.append(mod)
                flat = torch.stack([m._buffers["num_batches_tracked"].to(eng.device) for m in nbt])
                for i, m in enumerate(nbt):
                    m._buffers["num_batches_tracked"] = flat[i]
                self._nbt, self._nbt_inc = flat, torch.ones_like(flat)
            self._alias_ptr = sentinel.data_ptr()
            self._dirty = True

    def inference_engine(self, capacity: int, T: int, H: int, W: int, device):
        """The cached forward-only eval engine (engine_ft.InferenceEngine) of this batch capacity and clip size.  It reads
        the parameters and BatchNorm running statistics of the bound engine; while no engine is bound, the first one
        created owns them and the parameters are aliased onto it, as _bind_ft does.
        A pretraining model gets an engine_ft.FeatureEngine instead: the online network up to its pooled feature, reading
        the live weights and running statistics of the bound step engine."""
        from ... import engine_ft
        if self.pretrain:
            return self._feature_engine(capacity, T, H, W, device)
        if not isinstance(self.cls_bn, nn.Module):
            raise TypeError("'bool' object is not callable")
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        owner = self._engine
        if owner is None:
            owner = self._infer_owner
            if owner is not None and owner.device != device:
                self.free_inference_engines()
                owner = None
        elif owner.device != device:
            raise _engine_mod.ops.L.CstpError(f"the bound engine lives on {owner.device}, not {device}")
        key = (capacity, T, H, W, device)
        eng = self._infer.get(key)
        if eng is None:
            eng = engine_ft.InferenceEngine(capacity, T, H, W, device=device, num_classes=self.num_classes, cls_bn=True,
                                            share=owner, **getattr(self, "engine_options", {}))
            self._infer[key] = eng
            if owner is None:
                self._infer_owner = owner = eng
                self._alias_ptr = None
        self._alias_ft(owner)
        return eng

    def _feature_engine(self, capacity, T, H, W, device):
        from ... import engine_ft
        eng = self._engine
        if eng is None:
            raise _engine_mod.ops.L.CstpError(
                "the features of a pretraining model are those of its live step engine: run train_step (or "
                "train.load_checkpoint with example_clip) before extracting them")
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if eng.device != device:
            raise _engine_mod.ops.L.CstpError(f"the bound engine lives on {eng.device}, not {device}")
        key = (capacity, T, H, W, device)
        feat = self._infer.get(key)
        if feat is None:
            opts = {k: v for k, v in getattr(self, "engine_options", {}).items()
                    if k in ("fuse_apply", "fuse_min_positions", "fuse_policy")}
            feat = self._infer[key] = engine_ft.FeatureEngine(capacity, T, H, W, device=device, share=eng, **opts)
        return feat

    def free_inference_engines(self):
        """Frees the cached eval engines of other batch sizes (activations, packed weights, CUDA graphs); the next eval
        forward builds what it needs again.  The bound training engine is not affected."""
        self._infer.clear()
        if self._infer_owner is not None:
            self._infer_owner = None
            if self._engine is None:
                self._alias_ptr = None          # the parameters move to the next engine that is built
        if self._last_engine is not self._engine:
            self._last_engine = None

    def _repack_if_changed(self, eng):
        """Re-packs eng's bf16 tensor-core weights when the fp32 parameters changed since it last packed them.  The
        parameters are views of the engines' shared flat buffer, so every in-place update (optimizer.step,
        load_state_dict) bumps the version counter of that buffer; every other change (the fused finetune step, edits
        announced through _dirty) starts a new weight generation."""
        if self._dirty:
            self._wgen += 1
            self._dirty = self.pretrain          # a pretraining model's step engine re-packs (and clears it) in train_step
        key = (eng.train.data._version, self._wgen)
        if getattr(eng, "_packed_key", None) != key:
            eng.pack_online()
            eng._packed_key = key

    def _forward_ft(self, x1):
        if not self.training:
            return self._forward_eval_ft(x1)
        eng = self._bind_ft(x1)
        self._last_engine = eng
        x1 = x1.contiguous()
        if torch.is_grad_enabled():
            out = _FinetuneFn.apply(self, x1, *self._trainable())
            self._nbt += self._nbt_inc
            self._dirty = True
            return out
        self._repack_if_changed(eng)
        eng.eval_mode = False
        eng.forward(x1)
        self._nbt += self._nbt_inc
        return eng.logits[:, :self.num_classes].clone()

    def _forward_eval_ft(self, x):
        """model.eval() forward.  A batch of the bound engine's geometry runs on that engine; any other batch size runs on
        the cached inference engine of its capacity bucket (engine_ft.inference_capacity), which leaves the bound engine,
        its momentum and its captured step untouched.  Logits are bit-identical either way."""
        from ... import engine_ft
        _engine_mod.ops.require_device(x)
        eng = self._engine
        n = x.shape[0]
        if eng is not None and (self._engine_key == self._ft_key(x) or eng.device != x.device):
            eng = self._bind_ft(x)
            self._repack_if_changed(eng)
            eng.forward_eval(x.contiguous())
        else:
            _, _, T, H, W = x.shape
            eng = self.inference_engine(engine_ft.inference_capacity(n), T, H, W, x.device)
            self._repack_if_changed(eng)
            eng.forward_batch(x)
        self._last_engine = eng
        return eng.logits[:n, :self.num_classes].clone()

    @torch.no_grad()
    def finetune_step(self, x, labels, lr=0.025, momentum=0.9, weight_decay=1e-3, grad_sync=None, optimizer="sgd",
                      betas=(0.9, 0.999), eps=1e-8):
        """One fused finetune step (main_ft_mp.py:196-214: forward, CrossEntropyLoss, backward, SGD.step -- no gradient
        clipping in the finetune driver).  optimizer="adam" / "adamw" steps torch.optim.Adam / AdamW(lr, betas, eps,
        weight_decay) instead, and `momentum` is unused.  Returns the device scalar loss without synchronising."""
        eng = self._bind_ft(x)
        eng.select_optimizer(optimizer)          # an invalid or conflicting kind raises before anything runs
        eng.eval_mode = False
        eng.forward(x.contiguous(), repack=self._dirty)
        self._dirty = False
        eng.cross_entropy(labels)
        if eng.backward(grad_sync):
            grad_sync.finish()
        elif grad_sync is not None:
            grad_sync(eng.grad)
        # parameters frozen by get_fine_tuning_parameters (requires_grad = False) are skipped like optim.SGD skips them
        frozen = frozenset(n for n, p in self.named_parameters() if not p.requires_grad)
        if frozen != getattr(self, "_ft_frozen", None) or getattr(self, "_ft_ranges_eng", None) is not eng:
            self._ft_frozen, self._ft_ranges_eng = frozen, eng
            self._ft_ranges = eng.trainable_ranges(frozen) if frozen else None
        eng.optimizer_step(lr, momentum, weight_decay, ranges=self._ft_ranges, optimizer=optimizer, betas=betas, eps=eps)
        self._nbt += self._nbt_inc
        self._wgen += 1                          # the kernel updated the weights: other engines must re-pack
        eng._packed_key = (eng.train.data._version, self._wgen)       # optimizer_step re-packed this one
        self._last_engine = eng
        return eng.loss

    def _bump_nbt(self):
        self._nbt += self._nbt_inc

    def mark_weights_dirty(self):
        """Call after changing parameters behind the engine's back (e.g. in-place edits) before a fused train_step."""
        self._dirty = True

    def load_state_dict(self, *a, **k):
        r = super().load_state_dict(*a, **k)
        self._dirty = True
        return r

    # ------------------------------------------------------------------------------------------ reference interface
    def forward(self, x1, x2=None, o_type=None):
        if o_type in ("ft_fc", "ft_all", "test") and not self.pretrain:
            return self._forward_ft(x1)
        if o_type == "loss_com" and self.pretrain:
            self._bind(x1)
            outs = _LossComFn.apply(self, x1.contiguous(), x2.contiguous(), *self._trainable())
            self._nbt += self._nbt_inc
            self._dirty = True
            return outs[0], tuple(outs[1:])
        if o_type in ("r_byol", "ft_fc", "ft_all", "test", "loss_com"):
            raise NotImplementedError(f"o_type={o_type!r} with pretrain={self.pretrain}: 'loss_com' needs the pretraining "
                                      "model, 'ft_fc'/'ft_all'/'test' the finetune model (r_byol is broken in the reference "
                                      "itself, SURVEY.md 0.9)")
        raise ValueError("Output cls is not exist!")

    def _trainable(self):
        if getattr(self, "_trainable_cache", None) is None:
            named = dict(self.named_parameters())
            self._trainable_cache = [named[n] for n in self._trainable_names]
        return self._trainable_cache

    # ------------------------------------------------------------------------------------------ fused fast path
    @torch.no_grad()
    def train_step(self, x1, x2, labels, loss_weight=(0.1, 1, 1, 1, 1), lr=0.03, momentum=0.9, weight_decay=5e-4,
                   clip_grad_norm=18.0, grad_sync=None, optimizer="sgd", betas=(0.9, 0.999), eps=1e-8,
                   collapse_stats=False):
        """One full pretraining step (main_byol.py:60-91) as a single launch program.  optimizer="adam" / "adamw" steps
        torch.optim.Adam / AdamW(lr, betas, eps, weight_decay) after the same gradient clipping; `momentum` is then unused.
        collapse_stats=True adds one launch right after the BYOL loss that writes the step's representation statistics
        (see step_stats); losses, gradients, weights and buffers are bit for bit those of a step without it.  A setting
        that differs from the captured step's drops that graph and captures the step again.

        labels = (spa, tem, pb, rot1, rot2) int64 device tensors.  `grad_sync(flat_grad)` is called between backward
        and the optimiser (data-parallel all-reduce).  Returns the engine's device loss vector
        [ce_spa, ce_tem, ce_pb1, ce_pb2, ce_rot1, ce_rot2, weighted CE sum, loss_byol] without synchronising."""
        eng = self._bind(x1)
        eng.select_optimizer(optimizer)          # an invalid or conflicting kind raises before anything runs
        if eng.collapse_stats != bool(collapse_stats):
            eng.collapse_stats = bool(collapse_stats)
            eng.drop_graph()
        self._wgen += 1                          # the step updates the weights in place: feature engines must re-pack
        if tuple(loss_weight) != getattr(self, "_lw", None):
            eng.set_loss_weight(loss_weight)
            self._lw = tuple(loss_weight)
        if self._dirty:
            eng.pack_online()
            self._dirty = False
        if eng.use_graph and eng._prof is None:
            # everything behind the input pass replayed from a CUDA graph (engine.graphed_step)
            eng.graphed_step(x1, x2, labels, lr, momentum, weight_decay, clip_grad_norm or 0.0, bool(clip_grad_norm),
                             grad_sync, self._bump_nbt, optimizer, betas, eps)
            return eng.losses
        eng.forward(x1, x2)
        eng.pretext_losses(labels)
        if eng.backward(grad_sync):
            grad_sync.finish()                   # the all-reduce ran in buckets beside the backward pass
        elif grad_sync is not None:
            grad_sync(eng.grad)
        eng.optimizer_step(lr, momentum, weight_decay, clip_grad_norm or 0.0, bool(clip_grad_norm), optimizer, betas, eps)
        self._nbt += self._nbt_inc
        return eng.losses

    def step_stats(self) -> torch.Tensor:
        """Representation statistics of the last train_step run with collapse_stats=True, as the bound engine's device
        tensor fp32 [2 views][5] (no synchronisation; the next such step overwrites it).  Columns, in order
        (ops.REPR_STATS): std_feat, std_proj, std_pred, std_tproj -- the mean over the 512 columns of the unbiased
        standard deviation over the view's samples of the l2-normalised online pooled feature, projector output,
        predictor output and target projector output (about 1/sqrt(512) = 0.0442 for well-spread embeddings, 0 for a
        collapsed, constant one) -- and feat_norm, the mean norm of the pooled feature."""
        if self._engine is None or not self.pretrain:
            raise RuntimeError("step_stats() belongs to a pretraining model that has run train_step")
        return self._engine.step_stats
