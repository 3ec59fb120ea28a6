"""Class activation maps (Grad-CAM) and input saliency of a finetuned action classifier.

    result = class_activation_maps(model, clips, classes=None, stage="conv5", input_grad=False)

For an R21DBYOL(pretrain=False) in eval semantics (running statistics everywhere, whatever model.training is):

    logits     = classify(cls_bn(F.normalize(online_net(clips))))
    k          = classes, or logits.argmax(1) (ties to the lower class)
    score      = logits.gather(1, k[:, None]).sum()          eval BatchNorm couples no clips: one backward serves all
    A, dA      = the output of `stage` (block output after its ReLU) and d score / dA
    alpha      = dA.mean over (t, h, w);  cam = relu(sum_c alpha_c * A_c)
    cam        = trilinear upsampling to the clip (align_corners=False), min-max normalised per clip (zeros when flat)
    input_grad = d score / d clips (with input_grad=True)

Everything runs on the B200 (engine_ft.ExplainEngine): the eval forward of the inference engines, whose logits are
bit-identical to the model's eval forward, an eval-mode backward program with data gradients only, and the Grad-CAM
kernels of csrc/explain.cu.  Nothing of the model changes: no parameter, running statistic, num_batches_tracked, optimiser
state or other engine's captured graph, and no random generator is drawn from.
"""
from __future__ import annotations

from typing import NamedTuple

import torch

from . import engine as E
from .engine_ft import EXPLAIN_STAGES, inference_capacity

EXPLAIN_CHUNK = 64       # clips per engine run: larger batches run in chunks of at most this many clips


class CamResult(NamedTuple):
    logits: torch.Tensor              # fp32 [n][num_classes]
    classes: torch.Tensor             # int64 [n]: the explained class of every clip
    cam: torch.Tensor                 # fp32 [n][T][H][W], in [0, 1]
    input_grad: torch.Tensor | None   # fp32 [n][3][T][H][W] with input_grad=True


def class_activation_maps(model, clips: torch.Tensor, classes=None, *, stage: str = "conv5",
                          input_grad: bool = False) -> CamResult:
    """Grad-CAM maps of `stage` ("conv2" .. "conv5") for fp32 clips (n, 3, T, H, W) on the model's device, explaining
    `classes` (n class indices) or each clip's predicted class; see the module docstring.  `model` is a finetune
    R21DBYOL, bare or DDP-wrapped."""
    from .models.pace.r21d_byol import R21DBYOL
    from .train import unwrap
    m = unwrap(model)
    if not isinstance(m, R21DBYOL) or m.pretrain:
        raise ValueError("class activation maps need a finetune model, R21DBYOL(pretrain=False): a pretraining model has "
                         "no class score")
    if stage not in EXPLAIN_STAGES:
        raise ValueError(f"stage {stage!r}: expected one of {EXPLAIN_STAGES}")
    if not isinstance(clips, torch.Tensor) or clips.dim() != 5 or clips.shape[1] != 3 or clips.shape[0] < 1:
        raise ValueError(f"clips must be a (n, 3, T, H, W) tensor with n >= 1, got "
                         f"{tuple(clips.shape) if isinstance(clips, torch.Tensor) else type(clips).__name__}")
    if clips.dtype != torch.float32:
        raise TypeError(f"clips must be float32, got {clips.dtype}")
    E.ops.require_device(clips)
    n, _, T, H, W = clips.shape
    if H % 2 or W % 4:
        raise ValueError(f"clips of {H} x {W}: the stem needs an even height and a width that is a multiple of 4")
    if classes is not None:
        classes = torch.as_tensor(classes)
        if classes.dim() != 1 or classes.shape[0] != n or classes.dtype.is_floating_point or classes.dtype == torch.bool:
            raise ValueError(f"classes must hold one integer class per clip ({n}), got {classes.dtype} "
                             f"{tuple(classes.shape)}")
        lo, hi = int(classes.min()), int(classes.max())
        if lo < 0 or hi >= m.num_classes:
            raise ValueError(f"classes must lie in [0, {m.num_classes}), got values in [{lo}, {hi}]")
        classes = classes.to(device=clips.device, dtype=torch.int64)
    x = clips.contiguous()
    out_logits, out_classes, out_cam, out_dx = [], [], [], []
    for s in range(0, n, EXPLAIN_CHUNK):
        e = min(n, s + EXPLAIN_CHUNK)
        eng = m.explain_engine(inference_capacity(e - s), T, H, W, x.device, stage, input_grad)
        m._repack_if_changed(eng)
        eng.run(x[s:e], None if classes is None else classes[s:e])
        out_logits.append(eng.logits[:e - s, :m.num_classes].clone())
        out_classes.append(eng.classes[:e - s].clone())
        out_cam.append(eng.cam[:e - s].clone())
        if input_grad:
            out_dx.append(eng.dx[:e - s].clone())
    return CamResult(torch.cat(out_logits), torch.cat(out_classes), torch.cat(out_cam),
                     torch.cat(out_dx) if input_grad else None)
