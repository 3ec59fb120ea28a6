"""The JPEG decoder's stand-in (tests/emulate_jpeg.py, the kernels' integer arithmetic) against Pillow, byte for byte,
over a fixture matrix generated here; the rejection codes; `jpeg_size`; and the host logic of the JPEG-fed batch
source (distinct frames, slab remap, random draws identical to `PretrainBatches`)."""
import random
from functools import lru_cache

import numpy as np
import pytest
import torch
from PIL import features

from cstp_b200.data_process.datasets import JpegPretrainBatches, PretrainBatches, distinct_frames
from cstp_b200.data_process.jpeg import jpeg_size
from tests import emulate_jpeg as E
from tests import jpeg_cases as J

pytestmark = pytest.mark.skipif(not features.check_feature("libjpeg_turbo"),
                                reason="the decode contract is Pillow on libjpeg-turbo")


@lru_cache(maxsize=1)
def _good():
    return J.good_cases()


@lru_cache(maxsize=1)
def _bad():
    return J.bad_cases()


def test_matrix_covers_the_contract():
    names = [c[0] for c in _good()]
    for tag in ("1x1", "7x5", "15x17", "16x16", "33x47", "171x128", "340x256", "_444_", "_422_", "_420_", "_gray_",
                "q1_", "q50_", "q75_", "q95_", "q100_", "optimize", "rst_blocks1", "rst_blocks3", "rst_rows1", "cv2_",
                "split_tables", "merged_tables", "tables_after_sof", "app_com", "fill_bytes", "dqt16_sof1"):
        assert any(tag in n for n in names), tag


@pytest.mark.parametrize("i", range(len(J.good_cases(full=True))))
def test_stand_in_equals_pillow(i):
    name, b, w, h = _good()[i]
    status, out = E.decode(b, w, h)
    assert status == E.OK, name
    ref = J.pillow_decode(b)
    assert out.shape == ref.shape and np.array_equal(out, ref), name


def test_idct_limits_follow_pillow():
    """Quantisation tables scaled far past what an encoder writes drive the IDCT into libjpeg-turbo's 16-bit wrap and
    saturation; the stand-in follows Pillow there too."""
    base = J.pil_encode(J.content("noise", 32, 32), "444", quality=100)
    p = base.index(b"\xff\xdb")
    seg = (base[p + 2] << 8) | base[p + 3]
    for scale in (4, 16, 64, 255):
        b = bytearray(base)
        q = p + 4
        while q < p + 2 + seg:
            b[q + 1:q + 65] = bytes([scale]) * 64
            q += 65
        status, out = E.decode(bytes(b), 32, 32)
        assert status == E.OK and np.array_equal(out, J.pillow_decode(bytes(b))), scale


@pytest.mark.parametrize("i", range(len(J.bad_cases())))
def test_stand_in_rejects(i):
    name, b, w, h, expected = _bad()[i]
    status, out = E.decode(b, w, h)
    if expected is None:
        assert status == E.MALFORMED or (status == E.OK and np.array_equal(out, J.pillow_decode(b))), name
    else:
        assert status == expected, (name, status)


def test_jpeg_size():
    for name, b, w, h in _good():
        assert jpeg_size(b) == (w, h), name
    b = J.pil_encode(J.content("video", 41, 23), "420", quality=70)
    assert jpeg_size(b) == (41, 23)
    for bad in (b"", b"\x89PNG\r\n", b[:20]):
        with pytest.raises(ValueError):
            jpeg_size(bad)


class _ShapeStore:
    """Stand-in for GpuVideoStore that only answers shapes (what PretrainBatches reads to plan a batch)."""
    device = torch.device("cpu")

    def __init__(self, sizes, counts):
        self.sizes, self.counts = sizes, counts

    def __getitem__(self, i):
        w, h = self.sizes[i]
        return torch.empty((1, 1, 1, 3), dtype=torch.uint8).expand(self.counts[i], h, w, 3)


def _seed(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


@pytest.mark.parametrize("variant", ["ucf", "kinetics"])
def test_batch_source_plans_like_pretrain_batches(variant):
    sizes = [(171, 128), (161, 121), (173, 131), (340, 256)]
    counts = [40, 57, 33, 64]
    reads = []

    def read_frames(video, frames):
        reads.append((video, list(frames)))
        return [b""] * len(frames)

    ref = PretrainBatches(_ShapeStore(sizes, counts), counts, 4, variant=variant)
    src = JpegPretrainBatches(read_frames, counts, 4, variant=variant, sizes=sizes, device="cpu")
    ids = [2, 0, 3, 1]
    for trial in range(3):
        _seed(trial)
        plans_ref, _ = ref._videos(ids)
        state_ref = (random.random(), np.random.rand(), torch.rand(1).item())
        _seed(trial)
        plans, frames = src._plan(ids)
        state = (random.random(), np.random.rand(), torch.rand(1).item())
        assert state == state_ref                       # the same random draws, in the same order
        for p, pr, fr in zip(plans, plans_ref, frames):
            assert p.labels() == pr.labels() and p.frame_base == pr.frame_base
            assert fr == sorted(set(fr)) and set(fr) == {f for v in pr.views for f in v.frames}
            for v, vr in zip(p.views, pr.views):
                assert [fr[k - p.frame_base] for k in v.frames] == vr.frames      # slab index -> original frame
                assert (v.rot, v.box, v.base, v.flip, v.angle, v.jitter, v.gray, v.blur_sigma) == \
                    (vr.rot, vr.box, vr.base, vr.flip, vr.angle, vr.jitter, vr.gray, vr.blur_sigma)
    assert not reads                                    # sizes given: no frame read to plan


def test_distinct_frames_of_the_kinetics_second_view():
    from cstp_b200.data_process.clip_plan import PretrainClipSampler
    _seed(5)
    plan = PretrainClipSampler(16, 112, "kinetics").plan(80, 340, 256)
    frames, remapped = distinct_frames(plan)
    assert len(frames) <= 32 and frames == sorted(set(frames))
    assert all(0 <= k < len(frames) for v in remapped.views for k in v.frames)


def test_frame_size_reads_the_first_frame_once():
    b = J.pil_encode(J.content("video", 45, 31), "420", quality=80)
    calls = []

    def read_frames(video, frames):
        calls.append((video, list(frames)))
        return [b] * len(frames)

    for variant, first in (("ucf", 1), ("kinetics", 0)):
        calls.clear()
        src = JpegPretrainBatches(read_frames, [20], 1, variant=variant, device="cpu")
        assert src.frame_size(0) == (45, 31) and src.frame_size(0) == (45, 31)
        assert calls == [(0, [first])]


def test_frame_dir_reader(tmp_path):
    from cstp_b200.data_process.jpeg import FrameDirReader
    for v in range(2):
        d = tmp_path / f"v_{v}"
        d.mkdir()
        for n in (1, 2, 3):
            (d / f"{n:05d}.jpg").write_bytes(bytes([v, n]))
        (d / f"img_{7:03d}.jpeg").write_bytes(b"x")
    r = FrameDirReader([str(tmp_path / "v_0"), str(tmp_path / "v_1")])
    assert r(1, [3, 1]) == [bytes([1, 3]), bytes([1, 1])]
    assert FrameDirReader([str(tmp_path / "v_0")], fmt="img_{:03d}.jpeg")(0, [7]) == [b"x"]
