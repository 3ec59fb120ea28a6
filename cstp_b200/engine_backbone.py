"""Backbone engine: R2Plus1DNet((1,1,1,1)).forward (models/pace/r21d_byol.py:215-229) on its own -- the backbone, the
average pool and, with `proj`, the projector -- over ONE BatchNorm statistics group, for the standalone
models.pace.r21d_byol.R2Plus1DNet module.

It reuses the builders every engine shares (ProgramEngine._backbone, ProgramEngine._mlp) and is built in three variants:

    grads=True                     train mode with a backward program: d feat (+ d proj) -> parameter gradients, and on
                                   request the gradient of the input clip (ops.stem_dgrad)
    grads=False                    train mode, forward only (a target network under torch.no_grad())
    grads=False, eval_mode=True    model.eval(): every BatchNorm is the affine map of its running statistics; a batch of
                                   any n <= B clips runs in rows [0, n)

Parameters live under the names of R21DBYOL's online network ("online_net.conv1.spatial_conv.weight", ...), so the unit
tags, the per-layer parity checker of the tests and the forward program are those of engine_ft.FeatureEngine and of
engine_ft.FinetuneEngine's backbone.  `share`: an engine whose parameter and BatchNorm running-statistics stores this one
reads (the module keeps one set of stores for all of its engines); the packed bf16 weights and everything else per call
(activations, statistics scratch, gradients) are this engine's own.
"""
from __future__ import annotations

import torch

from . import engine as E
from .engine import ProgramEngine, backbone_param_specs

PREFIX = "online_net"


class BackboneEngine(ProgramEngine):
    def __init__(self, B: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", *, proj: bool = False,
                 grads: bool = True, eval_mode: bool = False, share: "BackboneEngine | None" = None,
                 record: bool = False, overlap: bool = True, fuse_apply: bool | None = None,
                 fuse_min_positions: int | None = None, fuse_policy: str | None = None):
        if grads and eval_mode:
            raise ValueError("an eval-mode backbone engine is forward only")
        self.proj, self.grads = bool(proj), bool(grads)
        super().__init__(B, T, H, W, device, backbone_param_specs(PREFIX, project=self.proj), grads=self.grads,
                         share=share, record=record, overlap=bool(overlap) and self.grads, fuse_apply=fuse_apply,
                         fuse_min_positions=fuse_min_positions, fuse_policy=fuse_policy, graph=False)
        self.eval_mode = bool(eval_mode)
        self._build()

    # ------------------------------------------------------------------------------------------ build
    def _build(self):
        B = self.B
        f32 = dict(device=self.device, dtype=torch.float32)
        x5, bw_backbone = self._backbone(self.fwd_online, self.train, PREFIX, self.grads, "online")
        self.feat = torch.zeros(B, 512, **f32)
        self.feat_bf = self._act(B, 512) if self.proj else None
        self._rec("online.feat", self.feat)
        self.fwd_online.append(lambda: E.ops.avgpool_fwd(x5, self.feat, self.feat_bf))
        self.proj_out = None
        proj = None
        if self.proj:
            proj = self._mlp(self.fwd_online, self.train, self.grads, self.feat_bf, f"{PREFIX}.project.net", 512, 4096,
                             512, 1, tag="online.project")
            self.proj_out = proj["out_f32"]
        if not self.grads:
            self._finish_build()
            return
        # ---------------- backward program: projector (into dfeat, accumulating) -> pool -> backbone
        self.dfeat = torch.zeros(B, 512, **f32)
        self.dproj = torch.zeros(B, 512, **f32) if self.proj else None
        if proj is not None:
            self.bwd.append(proj["make_backward"](self.dproj, None, self.dfeat, True))
        d_x5 = self._dbuf(x5)
        self.bwd.append(lambda: E.ops.avgpool_bwd(self.dfeat, d_x5))
        self.bwd.extend(reversed(bw_backbone))
        self._stem_holder = bw_backbone[0].holder        # the stem unit's d(raw) (holder["g"]) after the backward pass
        self._finish_build()

    # ------------------------------------------------------------------------------------------ programs
    def forward(self, x: torch.Tensor) -> None:
        """fp32 NCDHW clips (n, 3, T, H, W), n <= B -> rows [0, n) of self.feat (and self.proj_out)."""
        n = x.shape[0]
        E.ops.stem_pack(x, self.stem_rows[:n])
        self._forward_program()

    def backward_from(self, dfeat, dproj=None, dx: torch.Tensor | None = None) -> None:
        """Backward program of the last forward: dfeat fp32 [B][512] (and dproj) -> self.grad (every parameter,
        overwritten); with dx (fp32 (B, 3, T, H, W)) also the gradient of the input clip."""
        if not self.grads:
            raise RuntimeError("this backbone engine was built without a backward program")
        if dfeat is None:
            self.dfeat.zero_()
        else:
            self.dfeat.copy_(dfeat)
        if self.proj:
            if dproj is None:
                self.dproj.zero_()
            else:
                self.dproj.copy_(dproj)
        self.backward()
        if dx is not None:
            self.input_grad(dx)

    def input_grad(self, dx: torch.Tensor) -> None:
        """d(clip) from the stem unit's d(raw) of the last backward pass (ops.stem_dgrad)."""
        E.ops.stem_dgrad(self._stem_holder["g"], self.train.view(f"{PREFIX}.conv1.spatial_conv.weight"), dx)
