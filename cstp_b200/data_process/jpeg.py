"""JPEG frames decoded on the GPU (csrc/jpeg_decode.cu), byte for byte what the reference gets from
`PIL.Image.open(path).convert("RGB")` on libjpeg-turbo (datasets.py:888, 1340-1345): only compressed bytes stay on the
host, and neither a resident store of decoded frames nor host cores for decoding are needed.

  * `jpeg_size(b)`       (width, height) from the SOF segment, read on the host without touching entropy data.
  * `GpuJpegDecoder`     `decode(streams, sizes, outs)`: one upload and one `cstp_jpeg_decode` call per batch on the
                         current stream; `check(status, names)` raises ValueError for the rejected images.
  * `FrameDirReader`     `read_frames(video, frame_numbers) -> [bytes]` for videos extracted to frame directories.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

from .. import lib as L
from .. import ops

REASONS = {L.CSTP_JPEG_UNSUPPORTED: "unsupported JPEG (progressive, arithmetic, lossless, 12-bit, CMYK / RGB, sampling "
                                    "other than 4:4:4 / 4:2:2 / 4:2:0 / grayscale, several scans or no Huffman table)",
           L.CSTP_JPEG_MALFORMED: "malformed or truncated JPEG stream",
           L.CSTP_JPEG_SIZE: "frame size differs from the expected size"}

_DESC = np.dtype({"names": [f for f, _ in L.JpegImage._fields_],
                  "formats": [np.int64, np.int64, np.uint64, np.int32, np.int32, np.int64],
                  "offsets": [getattr(L.JpegImage, f).offset for f, _ in L.JpegImage._fields_],
                  "itemsize": C.sizeof(L.JpegImage)})

_SOF = {0xC0, 0xC1, 0xC2, 0xC3, 0xC5, 0xC6, 0xC7, 0xC9, 0xCA, 0xCB, 0xCD, 0xCE, 0xCF}


def jpeg_size(b: bytes) -> Tuple[int, int]:
    """(width, height) of a JPEG stream: walks the marker segments by their lengths and stops at the first SOF."""
    n = len(b)
    if n < 4 or b[0] != 0xFF or b[1] != 0xD8:
        raise ValueError("not a JPEG stream (no SOI marker)")
    p = 2
    while True:
        if p >= n or b[p] != 0xFF:
            raise ValueError("malformed JPEG stream: no SOF segment")
        while p < n and b[p] == 0xFF:
            p += 1
        if p + 3 > n:
            raise ValueError("truncated JPEG stream before SOF")
        m, seg = b[p], (b[p + 1] << 8) | b[p + 2]
        if m in _SOF:
            if seg < 8 or p + 1 + seg > n:
                raise ValueError("truncated SOF segment")
            return (b[p + 6] << 8) | b[p + 7], (b[p + 4] << 8) | b[p + 5]
        if m == 0xDA or m == 0xD9 or seg < 2:
            raise ValueError("malformed JPEG stream: no SOF segment")
        p += 1 + seg


class GpuJpegDecoder:
    """Batched JPEG decoding into caller-provided CUDA uint8 [H][W][3] tensors on the current stream.

    The streams and their descriptors go through one of two pinned staging buffers and one host-to-device copy per call;
    a buffer is written only after the copy that last read it has completed (the pattern of
    `GpuClipPipeline._buffers`)."""

    def __init__(self, device="cuda"):
        self.device = torch.device(device)
        self._slots = [dict(host=None, dev=None, event=None), dict(host=None, dev=None, event=None)]
        self._turn = 0
        self._ws = None
        self._ws_bytes: Dict[Tuple[int, int], int] = {}

    def workspace_bytes(self, w: int, h: int) -> int:
        key = (int(w), int(h))
        if key not in self._ws_bytes:
            self._ws_bytes[key] = ops.jpeg_workspace_bytes(*key)
        return self._ws_bytes[key]

    def decode(self, streams: Sequence[bytes], sizes: Sequence[Tuple[int, int]], outs: Sequence[torch.Tensor]):
        """Decodes streams[i] (expected size sizes[i] = (w, h)) into outs[i]; returns the int32 status tensor on the
        device (0, or a CSTP_JPEG_* code per image).  Nothing here waits for the device."""
        if self.device.type != "cuda":
            raise L.CstpError("GpuJpegDecoder needs a CUDA device: JPEG decoding has no CPU fallback")
        n = len(streams)
        if n == 0 or len(sizes) != n or len(outs) != n:
            raise ValueError("one expected size and one output tensor per stream, at least one stream")
        lens = np.fromiter((len(b) for b in streams), dtype=np.int64, count=n)
        wh = np.asarray(sizes, dtype=np.int64).reshape(n, 2)
        for i, ((w, h), o) in enumerate(zip(sizes, outs)):
            if o.dtype != torch.uint8 or not self._on_device(o) or tuple(o.shape) != (h, w, 3) or not o.is_contiguous():
                raise ValueError(f"output {i} must be a contiguous uint8 tensor [{h}][{w}][3] on {self.device}")
        descs = np.zeros(n, dtype=_DESC)                  # cstp_jpeg_image, built column-wise
        descs["src_bytes"] = lens
        descs["src_offset"][1:] = np.cumsum(lens)[:-1]
        descs["out"] = [o.data_ptr() for o in outs]
        descs["width"], descs["height"] = wh[:, 0], wh[:, 1]
        ws_each = np.array([self.workspace_bytes(w, h) for w, h in sizes], dtype=np.int64)
        descs["ws_offset"][1:] = np.cumsum(ws_each)[:-1]
        ws = int(ws_each.sum())
        dsz = (descs.nbytes + 255) & ~255
        src = dsz + int(lens.sum())
        slot = self._slots[self._turn]
        self._turn ^= 1
        if slot["event"] is not None:
            slot["event"].synchronize()          # the upload that last read this staging buffer has completed
        if slot["host"] is None or slot["host"].numel() < src:
            cap = max(src, 2 * (slot["host"].numel() if slot["host"] is not None else 0))
            slot["host"] = torch.empty(cap, dtype=torch.uint8).pin_memory()
            slot["dev"] = torch.empty(cap, dtype=torch.uint8, device=self.device)
        hb = slot["host"].numpy()
        hb[:descs.nbytes] = descs.view(np.uint8)
        hb[dsz:src] = np.frombuffer(b"".join(bytes(b) for b in streams), dtype=np.uint8)
        slot["dev"][:src].copy_(slot["host"][:src], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        slot["event"] = ev
        if self._ws is None or self._ws.numel() < ws:
            self._ws = None
            self._ws = torch.empty(max(ws, 256), dtype=torch.uint8, device=self.device)
        status = torch.empty(n, dtype=torch.int32, device=self.device)
        ops.jpeg_decode(slot["dev"], dsz, n, status, self._ws)
        return status

    def _on_device(self, t: torch.Tensor) -> bool:
        return t.device.type == self.device.type and (self.device.index is None or t.device.index == self.device.index)

    @staticmethod
    def check(status, names: Sequence = None) -> None:
        """Raises ValueError naming the first rejected image (status: the device or host tensor `decode` returned)."""
        raise_for_status(status.cpu().numpy(), names)


def raise_for_status(status: np.ndarray, names: Sequence = None) -> None:
    bad = np.flatnonzero(status)
    if bad.size:
        i = int(bad[0])
        what = names[i] if names is not None else f"image {i}"
        more = f" ({bad.size - 1} more rejected in this batch)" if bad.size > 1 else ""
        raise ValueError(f"{what}: {REASONS.get(int(status[i]), f'status {int(status[i])}')}{more}")


class FrameDirReader:
    """read_frames for videos extracted to one directory of frame files each: frame number n of video v is
    `os.path.join(video_dirs[v], fmt.format(n))` -- `00001.jpg`, ... for the reference's UCF101 layout (frame numbers
    are 1-based there, clip_plan.py)."""

    def __init__(self, video_dirs: Sequence[str], fmt: str = "{:05d}.jpg"):
        self.video_dirs, self.fmt = list(video_dirs), fmt

    def __call__(self, video: int, frame_numbers: Sequence[int]) -> List[bytes]:
        out = []
        for n in frame_numbers:
            with open(os.path.join(self.video_dirs[video], self.fmt.format(n)), "rb") as f:
                out.append(f.read())
        return out
