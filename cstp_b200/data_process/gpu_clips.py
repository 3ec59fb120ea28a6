"""GPU execution of clip plans: decoded uint8 frames resident in HBM -> the (B, 3, T, S, S) fp32 clips x1 / x2 and the
collated pretext labels, i.e. what the reference's DataLoader hands to `train_BYOL` (main_byol.py:43-49).

Replaces the pixel half of (reference file:line) data_process/datasets.py:850-857, 888-932 and
data_process/preprocess_data.py:479-565, 1112-1122 (Pillow / torchvision on CPU worker processes).  The host part of
this module only turns a plan (cstp_b200/data_process/clip_plan.py) into the integer descriptors of
`cstp_clip_assemble` (include/cstp_b200.h): Pillow's resampling taps in Q22, the 16.16 affine coefficients of
`Image.rotate`, the Q24 weights of the box blur -- each computed with Pillow's own double / float arithmetic so that
the kernel's output equals the reference's clip bit for bit.  All pixel work runs in csrc/clip_pipeline.cu; there is
no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from functools import lru_cache
from typing import List, Sequence

import numpy as np
import torch

from .. import lib as L
from .clip_plan import SamplePlan, ViewPlan

KMAX = L.CSTP_CLIP_KMAX
PRECISION_BITS = 22
JITTER_CODE = {"brightness": 0, "contrast": 1, "saturation": 2, "hue": 3}


@lru_cache(maxsize=4096)
def resample_tables(in_size: int, out_size: int) -> np.ndarray:
    """Pillow's precompute_coeffs + normalize_coeffs_8bpc for BICUBIC over the whole axis (libImaging/Resample.c):
    int32 [out_size][2 + KMAX] = first source index, tap count, Q22 taps.  Double arithmetic in Pillow's order."""
    scale = in_size / out_size
    fscale = scale if scale >= 1.0 else 1.0
    support = 2.0 * fscale
    ksize = int(math.ceil(support)) * 2 + 1
    if ksize > KMAX:
        raise ValueError(f"crop side {in_size} needs {ksize} resampling taps per output pixel (limit {KMAX})")
    ss = 1.0 / fscale
    xx = np.arange(out_size, dtype=np.float64)
    center = (xx + 0.5) * scale
    xmin = np.trunc(center - support + 0.5).astype(np.int64)
    xmin[xmin < 0] = 0
    xmax = np.trunc(center + support + 0.5).astype(np.int64)
    xmax[xmax > in_size] = in_size
    cnt = xmax - xmin
    X = np.arange(ksize, dtype=np.int64)[None, :] + xmin[:, None]
    arg = ((X.astype(np.float64) - center[:, None]) + 0.5) * ss
    a = -0.5
    ax = np.abs(arg)
    inner = ((a + 2.0) * ax - (a + 3.0)) * ax * ax + 1
    outer = (((ax - 5) * ax + 8) * ax - 4) * a
    k = np.where(ax < 1.0, inner, np.where(ax < 2.0, outer, 0.0))
    valid = np.arange(ksize)[None, :] < cnt[:, None]
    k = np.where(valid, k, 0.0)
    ww = np.zeros(out_size, dtype=np.float64)
    for j in range(ksize):                        # sequential accumulation, as the C loop does
        ww = np.where(valid[:, j], ww + k[:, j], ww)
    k = np.where((ww != 0.0)[:, None], k / np.where(ww != 0.0, ww, 1.0)[:, None], k)
    q = k * float(1 << PRECISION_BITS)
    q = np.where(k < 0, np.trunc(q - 0.5), np.trunc(q + 0.5))
    tab = np.zeros((out_size, 2 + KMAX), dtype=np.int32)
    tab[:, 0] = xmin
    tab[:, 1] = cnt
    tab[:, 2:2 + ksize] = np.where(valid, q, 0.0).astype(np.int32)
    tab.setflags(write=False)
    return tab


def rotate_fixed(angle: float, w: int, h: int):
    """Image.rotate(angle) (NEAREST, centre (w/2, h/2), no expand) as libImaging/Geometry.c affine_fixed walks it:
    source x = (a2 + x*a0 + y*a1) >> 16, source y = (a5 + x*a3 + y*a4) >> 16.  None when the rotation is the identity."""
    angle = angle % 360.0
    if angle == 0.0:
        return None
    if angle in (90.0, 180.0, 270.0):
        raise NotImplementedError("Image.rotate by an exact multiple of 90 degrees takes Pillow's transpose path")
    cx, cy = w / 2.0, h / 2.0
    rad = -math.radians(angle)
    m = [round(math.cos(rad), 15), round(math.sin(rad), 15), 0.0, round(-math.sin(rad), 15), round(math.cos(rad), 15), 0.0]
    m[2] = m[0] * -cx + m[1] * -cy + m[2]
    m[5] = m[3] * -cx + m[4] * -cy + m[5]
    m[2] += cx
    m[5] += cy

    def fix(v):
        return int(math.floor(v * 65536.0 + 0.5))
    return (fix(m[0]), fix(m[1]), fix(m[2] + m[0] * 0.5 + m[1] * 0.5), fix(m[3]), fix(m[4]), fix(m[5] + m[3] * 0.5 + m[4] * 0.5))


def blur_params(sigma: float, size: int, passes: int = 3):
    """ImageFilter.GaussianBlur(radius=sigma) -> (radius, edge_a, edge_b, ww, fw) of libImaging/BoxBlur.c (float32
    arithmetic of _gaussian_blur_radius and ImagingHorizontalBoxBlur); None when the box radius is 0."""
    f = np.float32
    r = f(sigma)
    sigma2 = f(r * r / f(passes))
    big_l = f(math.sqrt(12.0 * float(sigma2) + 1.0))
    sm_l = f(math.floor((float(big_l) - 1.0) / 2.0))
    a = f((f(2) * sm_l + f(1)) * (sm_l * (sm_l + f(1)) - f(3) * sigma2))
    a = f(a / (f(6) * (sigma2 - (sm_l + f(1)) * (sm_l + f(1)))))
    fr = f(sm_l + a)
    if fr == 0:
        return None
    radius = int(fr)
    ww = int(f(1 << 24) / (fr * f(2) + f(1)))
    fw = ((1 << 24) - (radius * 2 + 1) * ww) // 2
    return radius, min(radius + 1, size), max(size - radius - 1, 0), ww, fw


def compile_view(view: ViewPlan, frame_base: int, W: int, H: int, S: int, video_ptr: int = 0, out_ptr: int = 0,
                 coef_ptr: int = 0):
    """ViewPlan -> (cstp_clip_view, int32 coefficient tables [2][S][2 + KMAX], crop height)."""
    d = L.ClipView()
    d.video, d.out, d.coef = video_ptr, out_ptr, coef_ptr
    d.W, d.H = W, H
    if len(view.frames) > L.CSTP_CLIP_T:
        raise ValueError("clip longer than CSTP_CLIP_T frames")
    for i, n in enumerate(view.frames):
        d.frames[i] = n - frame_base
    d.rot = view.rot
    x0, y0, x1, y1 = view.box
    for i, b in enumerate(view.box):
        d.box[i] = b
    d.flip = int(view.flip)
    for i in range(L.CSTP_CLIP_T):
        d.gray[i] = -1
    if view.base:
        fx = rotate_fixed(view.angle, S, S)
        if fx is not None:
            d.rotate = 1
            for i, c in enumerate(fx):
                d.rot_fix[i] = c
        if view.jitter is not None:
            d.n_jitter = len(view.jitter)
            for i, (name, factor) in enumerate(view.jitter):
                d.jitter_op[i] = JITTER_CODE[name]
                if name == "hue":
                    d.hue_shift = int(np.int32(factor * 255).astype(np.uint8))     # torchvision _functional_pil.adjust_hue
                else:
                    d.jitter_f[i] = factor
        if view.gray is not None:
            for i, c in enumerate(view.gray):
                d.gray[i] = c
        if view.blur_sigma is not None:
            bp = blur_params(view.blur_sigma, S)
            if bp is not None:
                d.blur = 1
                d.blur_radius, d.blur_edge_a, d.blur_edge_b, d.blur_ww, d.blur_fw = bp
    if view.resize is not None:
        # ClipScale + ClipCenterCrop: the WHOLE (unrotated) frame is resized to (ow, oh) and the S x S crop of the result is
        # rows x0.. / y0.. of Pillow's tap tables for that resize -- the kernel reads the full frame through them
        ow, oh = view.resize
        if view.rot != 0 or x1 - x0 != S or y1 - y0 != S or x0 < 0 or y0 < 0 or x1 > ow or y1 > oh:
            raise ValueError("resize views crop an S x S window inside the resized, unrotated frame")
        coef = np.stack([resample_tables(W, ow)[x0:x1], resample_tables(H, oh)[y0:y1]])
        for i, b in enumerate((0, 0, W, H)):
            d.box[i] = b
        return d, coef, H
    coef = np.stack([resample_tables(x1 - x0, S), resample_tables(y1 - y0, S)])
    return d, coef, y1 - y0


def clip_layout(S: int, max_crop_h: int):
    """(CTAs per (frame, view), shared-memory bytes per CTA) that `cstp_clip_assemble` launches for clips of side S whose
    tallest crop has max_crop_h rows: 1 CTA while the crop rows and two S x S images fit, else a cluster pair.  Raises
    CstpError, naming the crop height, when neither fits.  Host arithmetic only; needs no GPU."""
    cluster, smem = C.c_int(), C.c_int()
    L.check(L.load().cstp_clip_layout(int(S), int(max_crop_h), C.byref(cluster), C.byref(smem)))
    return cluster.value, smem.value


def collate_labels(plans: Sequence[SamplePlan], device=None):
    """default_collate of the per-sample label lists: [spa (B,), tem (B,), pb (B,), [rot1 (B,), rot2 (B,)]] int64
    (datasets.py:856-857, consumed at main_byol.py:45-49)."""
    def t(vals):
        x = torch.tensor(list(vals), dtype=torch.int64)
        return x.to(device, non_blocking=True) if device is not None else x
    return [t(p.spa_label for p in plans), t(p.tem_label for p in plans), t(p.pb_label for p in plans),
            [t(p.rot_labels[0] for p in plans), t(p.rot_labels[1] for p in plans)]]


class GpuClipPipeline:
    """assemble(plans, videos) -> (x1, x2): one `cstp_clip_assemble` launch per batch.

    videos[b]: CUDA uint8 tensor [F][H][W][3], contiguous; videos[b][i] is the frame the reference opens as number
    `plan.frame_base + i` (file 00001.jpg for UCF, list entry 0 for the Kinetics LMDB records)."""

    def __init__(self, sample_duration: int = 16, sample_size: int = 112, device="cuda"):
        self.T, self.S = int(sample_duration), int(sample_size)
        self.device = torch.device(device)
        self._stage = {}            # batch size -> (pinned descriptor bytes, pinned tables, device copies, event)

    def _buffers(self, n_views: int):
        if n_views not in self._stage:
            dsz = C.sizeof(L.ClipView)
            self._stage[n_views] = dict(
                hdesc=torch.empty(n_views * dsz, dtype=torch.uint8).pin_memory(),
                hcoef=torch.empty((n_views, 2, self.S, 2 + KMAX), dtype=torch.int32).pin_memory(),
                ddesc=torch.empty(n_views * dsz, dtype=torch.uint8, device=self.device),
                dcoef=torch.empty((n_views, 2, self.S, 2 + KMAX), dtype=torch.int32, device=self.device),
                event=None)
        return self._stage[n_views]

    def assemble_clips(self, plans, videos: List[torch.Tensor], out=None):
        """Finetune / validation / test clips (clip_plan.ClipPlan, one view each) -> (B, 3, T, S, S) fp32."""
        class _One:                      # a ClipPlan as a one-view SamplePlan for the shared descriptor path
            def __init__(self, p):
                self.views, self.frame_base = (p.view,), p.frame_base
        B = len(plans)
        if out is None:
            out = torch.empty((B, 3, self.T, self.S, self.S), dtype=torch.float32, device=self.device)
        self._assemble([_One(p) for p in plans], videos, (out,))
        return out

    def assemble(self, plans: List[SamplePlan], videos: List[torch.Tensor], out=None):
        B = len(plans)
        if out is None and self.device.type == "cuda":
            out = (torch.empty((B, 3, self.T, self.S, self.S), dtype=torch.float32, device=self.device),
                   torch.empty((B, 3, self.T, self.S, self.S), dtype=torch.float32, device=self.device))
        self._assemble(plans, videos, out)
        return out

    def _assemble(self, plans, videos: List[torch.Tensor], outs):
        if self.device.type != "cuda":
            raise L.CstpError("GpuClipPipeline needs a CUDA device: the clip pipeline has no CPU fallback")
        B = len(plans)
        if len(videos) != B:
            raise ValueError("one video tensor per plan")
        nv = len(outs)
        buf = self._buffers(nv * B)
        if buf["event"] is not None:
            buf["event"].synchronize()          # the previous batch's descriptor upload has left the pinned staging
        descs = (L.ClipView * (nv * B))()
        clip_bytes = 3 * self.T * self.S * self.S * 4
        coef_bytes = 2 * self.S * (2 + KMAX) * 4
        max_h = 0
        for b, (plan, vid) in enumerate(zip(plans, videos)):
            if vid.dtype != torch.uint8 or vid.device != outs[0].device or vid.dim() != 4 or vid.shape[3] != 3 or not vid.is_contiguous():
                raise ValueError("videos must be contiguous CUDA uint8 tensors [F][H][W][3]")
            F_, H, W, _ = vid.shape
            if len(plan.views) != nv:
                raise ValueError("plan and output disagree on the number of views")
            for v, (view, dst) in enumerate(zip(plan.views, outs)):
                if len(view.frames) != self.T:
                    raise ValueError("plan and pipeline disagree on sample_duration")
                lo, hi = min(view.frames) - plan.frame_base, max(view.frames) - plan.frame_base
                if lo < 0 or hi >= F_:
                    raise ValueError(f"plan reads frame {hi + plan.frame_base} of a {F_}-frame video")
                i = nv * b + v
                d, coef, ch = compile_view(view, plan.frame_base, W, H, self.S, vid.data_ptr(), dst.data_ptr() + b * clip_bytes,
                                           buf["dcoef"].data_ptr() + i * coef_bytes)
                descs[i] = d
                buf["hcoef"][i] = torch.from_numpy(coef)
                max_h = max(max_h, ch)
        buf["hdesc"].copy_(torch.frombuffer(bytearray(bytes(descs)), dtype=torch.uint8))
        buf["ddesc"].copy_(buf["hdesc"], non_blocking=True)
        buf["dcoef"].copy_(buf["hcoef"], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        buf["event"] = ev
        L.check(L.load().cstp_clip_assemble(buf["ddesc"].data_ptr(), nv * B, self.T, self.S, max_h,
                                            torch.cuda.current_stream().cuda_stream))
