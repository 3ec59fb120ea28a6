"""Finetune / test engine: the `ft_fc` / `ft_all` / `test` branch of R21DBYOL.forward (models/pace/r21d_byol.py:394-399)
driven by main_ft_mp.py:179-289 (train / validation) and test.py:76-93 (multi-clip inference).

    logits = classify(cls_bn(F.normalize(online_net(x), p=2, dim=1)))            R21DBYOL(pretrain=False, num_classes, cls_bn)

Builds on cstp_b200.engine.ProgramEngine (the backbone program builder and every kernel of the pretraining engine)
with ONE view per sample (one BatchNorm statistics group) and no target network; adds the L2-normalise / BatchNorm1d /
Linear head, the n-way cross-entropy, and an eval mode in which every BatchNorm is the affine map of its running statistics
(model.eval()): forward only, no statistics kernels, nothing updated.
"""
from __future__ import annotations

import torch

from . import engine as E
from .engine import OptimizerEngine, ProgramEngine, backbone_param_specs, pad16


def finetune_param_specs(num_classes: int, cls_bn: bool):
    """Parameters of R21DBYOL(pretrain=False) in registration order (r21d_byol.py:293-299; SURVEY.md A.5)."""
    s = backbone_param_specs("online_net", project=False)
    s += [("classify.weight", (num_classes, 512)), ("classify.bias", (num_classes,))]
    if cls_bn:
        s += [("cls_bn.weight", (512,)), ("cls_bn.bias", (512,))]
    return s


def _build_classifier(eng, grads: bool, backbone_grads: bool, dgrad_to: str | None = None) -> None:
    """The program of `eng`: online_net -> avgpool -> F.normalize -> cls_bn -> classify, and with `grads` the head's
    backward into eng.grad (classify; with `backbone_grads` also cls_bn, the normalisation, the pool and the backbone).
    dgrad_to (without grads): an eval-mode, data-gradient-only backward program from eng.dlogits down to that level of
    ProgramEngine.DGRAD_LEVELS, with no parameter gradient (ExplainEngine)."""
    ops = E.ops
    B = eng.B
    f32 = dict(device=eng.device, dtype=torch.float32)
    explain = dgrad_to is not None
    x5, bw_backbone = eng._backbone(eng.fwd_online, eng.train, "online_net", backbone_grads, "online", dgrad_to=dgrad_to)
    C = eng.num_classes
    Cp = pad16(C)
    eng.feat = torch.zeros(B, 512, **f32)
    eng.norms = torch.zeros(B, **f32)
    eng.nfeat = eng._act(B, 512)                     # F.normalize(feat) as bf16 rows
    eng.hfeat = eng._act(B, 512) if eng.cls_bn else eng.nfeat
    eng.logits = torch.zeros(B, Cp, **f32)
    eng.dlogits = torch.zeros(B, Cp, **f32) if grads or explain else None
    eng.loss = torch.zeros(1, **f32)
    eng.ce_ws = torch.zeros(max(B, 16), **f32)
    wc, wct = eng._packed(eng.train, "classify.weight", grads or explain)
    bias = eng.train.slot("classify.bias")
    p_cls = ops.linear_plan(eng.hfeat, wc, None, out_f32=eng.logits, bias=bias)
    site = eng._site(eng.train, grads, "cls_bn", 512, 1, B) if eng.cls_bn else None
    eng._rec("head.feat", eng.feat)
    eng._rec("head.nfeat", eng.nfeat)
    eng._rec("head.hfeat", eng.hfeat)
    eng._rec("head.logits", eng.logits)

    def head_fwd():
        ops.avgpool_fwd(x5, eng.feat, None)
        ops.l2norm_fwd(eng.feat, eng.nfeat, eng.norms, 512)
        if site is not None:
            eng._bn_forward(eng.nfeat, site)
            ops.bn_apply(eng.nfeat, site.st, eng.hfeat, relu=False)
        p_cls.run()
    eng.fwd_online.append(head_fwd)
    if not grads and not explain:
        eng._finish_build()
        return

    # ---------------- backward program: head -> pool -> backbone
    g_out = eng._act(B, Cp)
    d_h = eng._act(B, 512)
    g_n = eng._act(B, 512) if eng.cls_bn else d_h
    eng.dfeat = torch.zeros(B, 512, **f32)
    if explain:
        pd_h = ops.linear_plan(g_out, wct, d_h)
        d_x5 = eng._dbuf(x5)

        def head_dgrad():
            ops.cast_pad(eng.dlogits, g_out, cols=C)
            pd_h.run()
            if site is not None:
                ops.bn_backward_eval(d_h, None, eng.nfeat, site.st, g_n)
            ops.l2norm_bwd(eng.feat, eng.norms, g_n, eng.dfeat, 512)
            ops.avgpool_bwd(eng.dfeat, d_x5)
        eng.bwd.append(head_dgrad)
        eng.bwd.extend(reversed(bw_backbone))
        eng._finish_build()
        return
    dWc = eng.train.view("classify.weight", eng.grad)
    dbc = eng.train.view("classify.bias", eng.grad)
    g1 = ops.ConvGeom((1, 1, 1))
    h5, go5 = eng.hfeat.view(1, 1, 1, B, 512), g_out.view(1, 1, 1, B, Cp)
    eng._wg_numel = max(eng._wg_numel, eng._wgrad_need(h5, go5, g1))
    pd_h = ops.linear_plan(g_out, wct, d_h)
    holder = {}
    eng._deferred.append(lambda: holder.__setitem__("wg", ops.wgrad_plan(h5, go5, g1, C, 512, eng._wg)))
    eng._rec("head.g_out", g_out)
    eng._rec("head.d_h", d_h)
    eng._rec("head.g_n", g_n)
    eng._rec("head.dfeat", eng.dfeat)
    d_x5 = eng._dbuf(x5)

    def head_bwd():
        ops.cast_pad(eng.dlogits, g_out, cols=C)
        ops.colsum(g_out, C, dbc)
        holder["wg"].run(dWc)
        if not backbone_grads:
            return
        pd_h.run()
        if site is not None:
            ops.bn_backward(d_h, None, eng.nfeat, site.st, site.gamma, site.dgamma, site.dbeta, g_n,
                            sync=eng.bn_sync)
        ops.l2norm_bwd(eng.feat, eng.norms, g_n, eng.dfeat, 512)
        ops.avgpool_bwd(eng.dfeat, d_x5)
    eng.bwd.append(head_bwd)
    if backbone_grads:
        eng.bwd.extend(reversed(bw_backbone))
    eng._finish_build()


class FinetuneEngine(OptimizerEngine):
    def __init__(self, B: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", num_classes: int = 101,
                 cls_bn: bool = True, record: bool = False, overlap: bool = True, backbone_grads: bool = True,
                 bn_sync=None, fuse_apply: bool | None = None, fuse_min_positions: int | None = None,
                 fuse_policy: str | None = None):
        self.num_classes, self.cls_bn, self.backbone_grads = num_classes, bool(cls_bn), backbone_grads
        super().__init__(B, T, H, W, device, finetune_param_specs(num_classes, self.cls_bn), record=record,
                         overlap=overlap, bn_sync=bn_sync, fuse_apply=fuse_apply, fuse_min_positions=fuse_min_positions,
                         fuse_policy=fuse_policy)
        _build_classifier(self, True, backbone_grads)

    # ------------------------------------------------------------------------------------------ programs
    def load_clip(self, x: torch.Tensor):
        E.ops.stem_pack(x, self.stem_rows)

    def forward(self, x, repack: bool = False):
        """logits (device fp32 [B][pad16(num_classes)], the first num_classes columns are valid)."""
        if repack:
            self.pack_online()
        self.load_clip(x)
        self._forward_program()
        return self.logits

    def forward_eval(self, x, use_graph: bool = True):
        """model.eval() forward.  The ~75 small launches of a batch-1 clip are launch-bound (1.2 ms eager), so the
        program behind the input pass is replayed from a CUDA graph (weights are re-packed outside the graph into the
        same buffers, so the graph survives weight updates)."""
        self.eval_mode = True
        self.load_clip(x)
        if use_graph:
            self._captured("eval", None, self._forward_program)
        else:
            self._forward_program()
        return self.logits

    def cross_entropy(self, labels):
        """nn.CrossEntropyLoss() of main_ft_mp.py:188,203 on the current logits; fills self.loss and self.dlogits."""
        E.ops.ce_loss(self.logits, labels, self.num_classes, self.loss, self.dlogits, self.ce_ws)

    def trainable_ranges(self, frozen_names) -> list[tuple[int, int]]:
        """(offset, length) runs of the flat buffer that hold the parameters NOT in `frozen_names`, merged where the
        slots are adjacent.  optim.SGD skips parameters without a gradient entirely -- no weight decay, no momentum
        (r21d_byol.py:10-35 sets requires_grad = False on everything but `classify` for ft_fc)."""
        runs: list[list[int]] = []
        for name, (off, _) in self.train.slots.items():
            if name in frozen_names:
                continue
            n = self.train.slot(name).numel()
            if runs and runs[-1][0] + runs[-1][1] == off:
                runs[-1][1] += n
            else:
                runs.append([off, n])
        return [(o, n) for o, n in runs]

    def optimizer_step(self, lr, momentum=0.9, wd=1e-3, max_norm=0.0, clip=False, ranges=None, optimizer="sgd",
                       betas=(0.9, 0.999), eps=1e-8):
        """SGD.step of main_ft_mp.py:117-121,212 (no gradient clipping in the finetune driver), or Adam / AdamW.step.
        `ranges` restricts the update to the trainable runs of the flat buffer (see trainable_ranges): the other
        parameters get no update, and their optimiser state stays zero; None updates every parameter."""
        if ranges is None:
            return super().optimizer_step(lr, momentum, wd, max_norm, clip, optimizer, betas, eps)
        if clip:
            raise E.ops.L.CstpError("gradient clipping over a partial parameter set is not part of the finetune path")
        self.select_optimizer(optimizer)
        if optimizer == "sgd":
            for off, n in ranges:
                E.ops.sgd_clip_step(self.train.data[off:off + n], self.grad[off:off + n], self.mom[off:off + n], lr,
                                    momentum, wd, 0.0, False, self.first_step, self.norm_out, self.sgd_ws)
        else:
            h = self._next_adam(lr, betas, eps, wd, 0.0, False)
            for off, n in ranges:
                E.ops.adam_clip_step(self.train.data[off:off + n], self.grad[off:off + n], self.exp_avg[off:off + n],
                                     self.exp_avg_sq[off:off + n], h, self.norm_out, self.sgd_ws)
        self.first_step = False
        self.pack_online()


def inference_capacity(n: int) -> int:
    """Batch capacity of the inference engine that runs an eval forward of n clips: the smallest power of two >= n up to
    64, then the next multiple of 64 -- a handful of engines covers every clip count of a test set."""
    if n < 1:
        raise ValueError(f"an eval forward needs at least one clip, got {n}")
    return 1 << (n - 1).bit_length() if n <= 64 else (n + 63) // 64 * 64


class InferenceEngine(ProgramEngine):
    """Forward-only eval engine (model.eval(): every BatchNorm is the affine map of its running statistics) of a fixed
    batch `capacity` that evaluates any n <= capacity clips: `run(n)` computes rows [0, n) of `x_static` and leaves the
    other rows unread.  Eval BatchNorm couples no samples and the forward convolutions have no split-K, so a clip's
    logits do not depend on the batch it runs in: they are bit-identical to FinetuneEngine(n).forward_eval's.

    share: an engine whose parameter and BatchNorm running-statistics stores this one reads (the module's bound training
    engine); None allocates them here.  Either way the packed bf16 weights are this engine's own (pack_online)."""

    def __init__(self, capacity: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", num_classes: int = 101,
                 cls_bn: bool = True, share: ProgramEngine | None = None, **options):
        self.num_classes, self.cls_bn = num_classes, bool(cls_bn)
        options["overlap"] = False              # one stream: there is no target network and no backward pass
        super().__init__(capacity, T, H, W, device, finetune_param_specs(num_classes, self.cls_bn), grads=False,
                         share=share, **options)
        self.capacity = capacity
        self.eval_mode = True
        self.x_static = torch.zeros(capacity, 3, T, H, W, device=self.device, dtype=torch.float32)
        self._build()

    def _build(self):
        _build_classifier(self, False, False)

    def run(self, n: int) -> torch.Tensor:
        """Eval forward of rows [0, n) of x_static; returns self.logits, whose rows [0, n) are valid.  The program behind
        the input pass is replayed from a CUDA graph (ProgramEngine._captured)."""
        if not 1 <= n <= self.capacity:
            raise ValueError(f"{n} clips do not fit an inference engine of capacity {self.capacity}")
        E.ops.stem_pack(self.x_static[:n], self.stem_rows[:n])
        self._captured("eval", None, self._forward_program)
        return self.logits

    def forward_batch(self, x: torch.Tensor) -> torch.Tensor:
        """Copies the clips x (n, 3, T, H, W) into x_static and runs them (see run)."""
        self.x_static[:x.shape[0]].copy_(x)
        return self.run(x.shape[0])

    def cross_entropy(self, labels):
        """nn.CrossEntropyLoss() over the rows of the last run (labels has one entry per row); fills self.loss."""
        n = labels.shape[0]
        E.ops.ce_loss(self.logits[:n], labels, self.num_classes, self.loss, None, self.ce_ws)


class FeatureEngine(InferenceEngine):
    """Forward-only eval engine of the online network alone: its program ends at the average pool (`feat`, fp32
    [capacity][512]); there is no F.normalize, cls_bn or classify.  It reads the `online_net.*` weights and BatchNorm
    running statistics by name from the stores of `share`, a pretraining StepEngine (nothing is copied), and packs its
    own bf16 weights.  The backbone program is InferenceEngine's, so the features are bit-identical to those of a
    finetune model holding the same online-network weights and running statistics."""

    def _build(self):
        x5, _ = self._backbone(self.fwd_online, self.train, "online_net", False, "online")
        self.feat = torch.zeros(self.B, 512, device=self.device, dtype=torch.float32)
        self.logits = None                       # no classification head: run() returns None
        self._rec("head.feat", self.feat)
        self.fwd_online.append(lambda: E.ops.avgpool_fwd(x5, self.feat, None))
        self._finish_build()


EXPLAIN_STAGES = ("conv2", "conv3", "conv4", "conv5")


class ExplainEngine(ProgramEngine):
    """Grad-CAM engine (cstp_b200.explain) of a fixed batch `capacity`: the InferenceEngine's eval forward, then the
    gradient of the score logits[b, k_b] (k_b given or the argmax) through an eval-mode, data-gradient-only backward
    program -- the one-hot seed, the classifier dgrad, the cls_bn running-statistics map, l2norm_bwd, avgpool_bwd and the
    backbone's dgrad closures down to the output of `stage` (or, with `input_grad`, to the stem's d(raw) and the clip) --
    then the class-activation map of that stage, upsampled to the clip and min-max normalised.  Eval BatchNorm couples no
    clips, so one backward pass serves every row.  There are no weight gradients, no BatchNorm statistics and no
    running-statistics writes; transposed weights are packed only for the units the backward pass runs.

    share: the engine whose parameter and running-statistics stores this one reads (as InferenceEngine)."""

    EVAL_BACKWARD = True

    def __init__(self, capacity: int, T: int = 16, H: int = 112, W: int = 112, stage: str = "conv5",
                 input_grad: bool = False, device="cuda", num_classes: int = 101, cls_bn: bool = True,
                 share: ProgramEngine | None = None, **options):
        if stage not in EXPLAIN_STAGES:
            raise ValueError(f"stage {stage!r}: expected one of {EXPLAIN_STAGES}")
        self.num_classes, self.cls_bn = num_classes, bool(cls_bn)
        self.stage, self.input_grad = stage, bool(input_grad)
        options["overlap"] = False
        super().__init__(capacity, T, H, W, device, finetune_param_specs(num_classes, self.cls_bn), grads=False,
                         share=share, **options)
        self.capacity = capacity
        self.eval_mode = True
        f32 = dict(device=self.device, dtype=torch.float32)
        self.x_static = torch.zeros(capacity, 3, T, H, W, **f32)
        self.classes_in = torch.zeros(capacity, device=self.device, dtype=torch.int64)
        self.classes = torch.zeros(capacity, device=self.device, dtype=torch.int64)
        _build_classifier(self, False, False, dgrad_to="input" if self.input_grad else stage)
        unit = next(u for u in self.units if u["tag"] == f"online.{stage}.block1.conv2.temporal")
        self.stage_act = unit["act"]                       # the block output after its ReLU
        self.stage_grad = self._dbuf(self.stage_act)       # its gradient, left by the backward program
        self.stage_channels = unit["cout"]
        N, t, h, w, _ = self.stage_act.shape
        self.alpha = torch.zeros(capacity, self.stage_channels, **f32)
        self.cam_small = torch.zeros(capacity, t, h, w, **f32)
        self.cam = torch.zeros(capacity, T, H, W, **f32)
        self.dx = torch.zeros(capacity, 3, T, H, W, **f32) if self.input_grad else None

    def _program(self, n: int, given: bool):
        ops = E.ops
        self._forward_program()
        ops.cam_seed(self.logits, n, self.num_classes, self.classes_in if given else None, self.classes, self.dlogits)
        for op in self.bwd:
            op()
        ops.gradcam(self.stage_act, self.stage_grad, n, self.stage_channels, self.alpha, self.cam_small)
        ops.cam_upsample(self.cam_small, n, self.cam)
        if self.input_grad:
            g = self.bwd[-1].holder["g"]                   # the stem unit's d(raw)
            ops.stem_dgrad(g[:n], self.train.view("online_net.conv1.spatial_conv.weight"), self.dx[:n])

    def run(self, x: torch.Tensor, classes: torch.Tensor | None = None) -> None:
        """Clips x (n, 3, T, H, W), n <= capacity, and optionally their classes (int64 [n], on the device) -> rows [0, n)
        of logits, classes, cam (and dx).  The program behind the input pass is replayed from a CUDA graph
        (ProgramEngine._captured), one per (n, classes given)."""
        n = x.shape[0]
        if not 1 <= n <= self.capacity:
            raise ValueError(f"{n} clips do not fit an explain engine of capacity {self.capacity}")
        self.x_static[:n].copy_(x)
        if classes is not None:
            self.classes_in[:n].copy_(classes)
        E.ops.stem_pack(self.x_static[:n], self.stem_rows[:n])
        given = classes is not None
        self._captured("explain", (n, given), lambda: self._program(n, given))
