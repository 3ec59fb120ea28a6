"""Finetune / test engine: the `ft_fc` / `ft_all` / `test` branch of R21DBYOL.forward (models/pace/r21d_byol.py:394-399)
driven by main_ft_mp.py:179-289 (train / validation) and test.py:76-93 (multi-clip inference).

    logits = classify(cls_bn(F.normalize(online_net(x), p=2, dim=1)))            R21DBYOL(pretrain=False, num_classes, cls_bn)

Reuses the backbone program builder and every kernel of the pretraining engine (cstp_b200.engine.StepEngine) with ONE
view per sample (one BatchNorm statistics group) and no target network; adds the L2-normalise / BatchNorm1d / Linear
head, the n-way cross-entropy, and an eval mode in which every BatchNorm is the affine map of its running statistics
(model.eval()): forward only, no statistics kernels, nothing updated.
"""
from __future__ import annotations

import torch

from . import engine as E
from .engine import FlatStore, StepEngine, backbone_param_specs, bn_buffer_specs, pad16


def finetune_param_specs(num_classes: int, cls_bn: bool):
    """Parameters of R21DBYOL(pretrain=False) in registration order (r21d_byol.py:293-299; SURVEY.md A.5)."""
    s = backbone_param_specs("online_net", project=False)
    s += [("classify.weight", (num_classes, 512)), ("classify.bias", (num_classes,))]
    if cls_bn:
        s += [("cls_bn.weight", (512,)), ("cls_bn.bias", (512,))]
    return s


class FinetuneEngine(StepEngine):
    VIEWS = 1
    FORWARD_ONLY = False             # InferenceEngine: no backward program, no gradient / momentum store

    def __init__(self, B: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", num_classes: int = 101,
                 cls_bn: bool = True, record: bool = False, overlap: bool = True, backbone_grads: bool = True,
                 bn_sync=None, fuse_apply: bool | None = None, fuse_min_positions: int | None = None,
                 fuse_policy: str | None = None):
        self.num_classes, self.cls_bn, self.backbone_grads = num_classes, bool(cls_bn), backbone_grads
        super().__init__(B, T, H, W, device=device, record=record, overlap=overlap, bn_sync=bn_sync, fuse_apply=fuse_apply,
                         fuse_min_positions=fuse_min_positions, fuse_policy=fuse_policy)

    def _make_stores(self):
        self._make_param_stores()
        self.grad = self.train.like()
        self.mom = self.train.like()

    def _make_param_stores(self):
        specs = finetune_param_specs(self.num_classes, self.cls_bn)
        self.train = FlatStore(specs, self.device)
        self.target = None
        self.bufs = FlatStore(bn_buffer_specs(specs), self.device)
        for name in self.bufs.slots:
            if name.endswith("running_var"):
                self.bufs.view(name).fill_(1.0)

    # ------------------------------------------------------------------------------------------ build
    def _build(self):
        ops = E.ops
        B = self.B
        f32 = dict(device=self.device, dtype=torch.float32)
        x5, bw_backbone = self._backbone(self.fwd_online, self.train, "online_net", self.backbone_grads, "online")
        C = self.num_classes
        Cp = pad16(C)
        self.feat = torch.zeros(B, 512, **f32)
        self.norms = torch.zeros(B, **f32)
        self.nfeat = self._act(B, 512)                     # F.normalize(feat) as bf16 rows
        self.hfeat = self._act(B, 512) if self.cls_bn else self.nfeat
        head_grads = not self.FORWARD_ONLY
        self.logits = torch.zeros(B, Cp, **f32)
        self.dlogits = torch.zeros(B, Cp, **f32) if head_grads else None
        self.loss = torch.zeros(1, **f32)
        self.ce_ws = torch.zeros(max(B, 16), **f32)
        wc, wct = self._packed(self.train, "classify.weight", head_grads)
        bias = self.train.slot("classify.bias")
        p_cls = ops.linear_plan(self.hfeat, wc, None, out_f32=self.logits, bias=bias)
        site = self._site(self.train, head_grads, "cls_bn", 512, 1, B) if self.cls_bn else None
        self._rec("head.feat", self.feat)
        self._rec("head.nfeat", self.nfeat)
        self._rec("head.hfeat", self.hfeat)
        self._rec("head.logits", self.logits)

        def head_fwd():
            ops.avgpool_fwd(x5, self.feat, None)
            ops.l2norm_fwd(self.feat, self.nfeat, self.norms, 512)
            if site is not None:
                if self.eval_mode:
                    ops.bn_eval_coeffs(site.st, site.gamma, site.beta, site.rm, site.rv, E.BN_EPS)
                else:
                    ops.bn_forward_stats(self.nfeat, site.st, site.gamma, site.beta, site.rm, site.rv, E.BN_EPS,
                                         E.BN_MOMENTUM, sync=self.bn_sync)
                ops.bn_apply(self.nfeat, site.st, self.hfeat, relu=False)
            p_cls.run()
        self.fwd_online.append(head_fwd)
        if not head_grads:
            self._finish_build()
            return

        # ---------------- backward program: head -> pool -> backbone
        g_out = self._act(B, Cp)
        d_h = self._act(B, 512)
        g_n = self._act(B, 512) if self.cls_bn else d_h
        self.dfeat = torch.zeros(B, 512, **f32)
        dWc = self.train.view("classify.weight", self.grad)
        dbc = self.train.view("classify.bias", self.grad)
        g1 = ops.ConvGeom((1, 1, 1))
        h5, go5 = self.hfeat.view(1, 1, 1, B, 512), g_out.view(1, 1, 1, B, Cp)
        self._wg_numel = max(self._wg_numel, self._wgrad_need(h5, go5, g1))
        pd_h = ops.linear_plan(g_out, wct, d_h)
        holder = {}
        self._deferred.append(lambda: holder.__setitem__("wg", ops.wgrad_plan(h5, go5, g1, C, 512, self._wg)))
        self._rec("head.g_out", g_out)
        self._rec("head.d_h", d_h)
        self._rec("head.g_n", g_n)
        self._rec("head.dfeat", self.dfeat)
        d_x5 = self._dbuf(x5)

        def head_bwd():
            ops.cast_pad(self.dlogits, g_out, cols=C)
            ops.colsum(g_out, C, dbc)
            holder["wg"].run(dWc)
            if not self.backbone_grads:
                return
            pd_h.run()
            if site is not None:
                ops.bn_backward(d_h, None, self.nfeat, site.st, site.gamma, site.dgamma, site.dbeta, g_n,
                                sync=self.bn_sync)
            ops.l2norm_bwd(self.feat, self.norms, g_n, self.dfeat, 512)
            ops.avgpool_bwd(self.dfeat, d_x5)
        self.bwd.append(head_bwd)
        if self.backbone_grads:
            self.bwd.extend(reversed(bw_backbone))
        self._finish_build()

    # ------------------------------------------------------------------------------------------ programs
    def load_clip(self, x: torch.Tensor):
        E.ops.stem_pack(x, self.stem_rows)

    def forward(self, x, repack: bool = False):
        """logits (device fp32 [B][pad16(num_classes)], the first num_classes columns are valid)."""
        if repack:
            self.pack_online()
        self.load_clip(x)
        for op in self.fwd_online:
            op()
        return self.logits

    def forward_eval(self, x, use_graph: bool = True):
        """model.eval() forward.  The ~75 small launches of a batch-1 clip are launch-bound (1.2 ms eager), so the
        program is captured once into a CUDA graph over a static input buffer and replayed (weights are re-packed outside
        the graph into the same buffers, so the graph survives weight updates)."""
        self.eval_mode = True
        if not use_graph or self.device.type != "cuda":
            return self.forward(x)
        if getattr(self, "_graph", None) is None:
            self._x_static = torch.empty_like(x)
            self._x_static.copy_(x)
            self.forward(self._x_static)                   # eager warm-up: one-time kernel attribute calls happen here
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self.forward(self._x_static)
            self._graph = g
        self._x_static.copy_(x)
        self._graph.replay()
        return self.logits

    def cross_entropy(self, labels):
        """nn.CrossEntropyLoss() of main_ft_mp.py:188,203 on the current logits; fills self.loss and self.dlogits."""
        E.ops.ce_loss(self.logits, labels, self.num_classes, self.loss, self.dlogits, self.ce_ws)

    def trainable_ranges(self, frozen_names) -> list[tuple[int, int]]:
        """(offset, length) runs of the flat buffer that hold the parameters NOT in `frozen_names`, merged where the
        slots are adjacent.  optim.SGD skips parameters without a gradient entirely -- no weight decay, no momentum
        (r21d_byol.py:10-35 sets requires_grad = False on everything but `classify` for ft_fc)."""
        runs: list[list[int]] = []
        for name, (off, shape) in self.train.slots.items():
            if name in frozen_names:
                continue
            n = 1
            for d in shape:
                n *= d
            n = (n + 15) // 16 * 16
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


class InferenceEngine(FinetuneEngine):
    """Forward-only eval engine (model.eval(): every BatchNorm is the affine map of its running statistics) of a fixed
    batch `capacity` that evaluates any n <= capacity clips: `run(n)` computes rows [0, n) of `x_static` and leaves the
    other rows unread.  Eval BatchNorm couples no samples and the forward convolutions have no split-K, so a clip's
    logits do not depend on the batch it runs in: they are bit-identical to FinetuneEngine(n).forward_eval's.

    share: an engine whose parameter and BatchNorm running-statistics stores this one reads (the module's bound training
    engine); None allocates them here.  Either way the packed bf16 weights are this engine's own (pack_online)."""

    FORWARD_ONLY = True

    def __init__(self, capacity: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", num_classes: int = 101,
                 cls_bn: bool = True, share: FinetuneEngine | None = None, **options):
        self._share = share
        options["overlap"] = False              # one stream: there is no target network and no backward pass
        super().__init__(capacity, T, H, W, device=device, num_classes=num_classes, cls_bn=cls_bn, backbone_grads=False,
                         **options)
        self.capacity = capacity
        self.eval_mode = True
        self.x_static = torch.zeros(capacity, 3, T, H, W, device=self.device, dtype=torch.float32)

    def _make_stores(self):
        if self._share is None:
            self._make_param_stores()
        else:
            self.train, self.bufs, self.target = self._share.train, self._share.bufs, None
        self.grad = self.mom = None

    def run(self, n: int) -> torch.Tensor:
        """Eval forward of rows [0, n) of x_static; returns self.logits, whose rows [0, n) are valid.  The program behind
        the input pass is replayed from a CUDA graph captured on the first call."""
        if not 1 <= n <= self.capacity:
            raise ValueError(f"{n} clips do not fit an inference engine of capacity {self.capacity}")
        E.ops.stem_pack(self.x_static[:n], self.stem_rows[:n])
        if not self.use_graph:
            for op in self.fwd_online:
                op()
            return self.logits
        if self._graph is None:
            for op in self.fwd_online:           # eager warm-up: one-time kernel attribute calls happen here
                op()
            torch.cuda.synchronize(self.device)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for op in self.fwd_online:
                    op()
            self._graph = g
        self._graph.replay()
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
