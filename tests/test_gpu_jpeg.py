"""GPU JPEG decoding (csrc/jpeg_decode.cu) against Pillow and the stand-in, byte for byte, in batches that mix sizes and
samplings; the rejection contract in a batch that mixes malformed and good streams; `GpuVideoStore.put_jpeg`; and the
JPEG-fed pretraining batches against `PretrainBatches` over a store of Pillow-decoded copies of the same frames."""
import random

import numpy as np
import pytest
import torch
from PIL import features

from cstp_b200.data_process.datasets import GpuVideoStore, JpegPretrainBatches, PretrainBatches
from cstp_b200.data_process.jpeg import GpuJpegDecoder
from tests import emulate_jpeg as E
from tests import jpeg_cases as J

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not features.check_feature("libjpeg_turbo"),
                                                  reason="the decode contract is Pillow on libjpeg-turbo")]


def _decode(dec, cases):
    outs = [torch.full((h, w, 3), 77, dtype=torch.uint8, device="cuda") for _, _, w, h in cases]
    status = dec.decode([c[1] for c in cases], [(c[2], c[3]) for c in cases], outs)
    return status.cpu().numpy(), [o.cpu().numpy() for o in outs]


def test_kernels_equal_pillow_over_the_matrix():
    cases = J.good_cases()
    order = list(range(len(cases)))
    random.Random(0).shuffle(order)                     # batches mix sizes, samplings and encoders
    dec = GpuJpegDecoder("cuda")
    bad = []
    for k in range(0, len(order), 61):
        batch = [cases[i] for i in order[k:k + 61]]
        status, outs = _decode(dec, batch)
        for (name, b, w, h), st, out in zip(batch, status, outs):
            if st != 0 or not np.array_equal(out, J.pillow_decode(b)):
                bad.append((name, int(st)))
    assert not bad, bad[:20]


def test_kernels_follow_the_idct_limits():
    base = J.pil_encode(J.content("noise", 32, 32), "444", quality=100)
    p = base.index(b"\xff\xdb")
    seg = (base[p + 2] << 8) | base[p + 3]
    cases = []
    for scale in (4, 16, 64, 255):
        b = bytearray(base)
        q = p + 4
        while q < p + 2 + seg:
            b[q + 1:q + 65] = bytes([scale]) * 64
            q += 65
        cases.append((f"scale{scale}", bytes(b), 32, 32))
    status, outs = _decode(GpuJpegDecoder("cuda"), cases)
    for (name, b, w, h), st, out in zip(cases, status, outs):
        assert st == 0 and np.array_equal(out, J.pillow_decode(b)), name
        assert np.array_equal(out, E.decode(b, w, h)[1]), name


def test_malformed_streams_mixed_with_good_ones():
    good = [c for c in J.good_cases() if c[2] * c[3] <= 171 * 128][::9]
    bad = J.bad_cases()
    mixed = []
    for i, c in enumerate(bad):
        mixed.append(("bad",) + c)
        mixed += [("good",) + g for g in good[i * 3:i * 3 + 3]]
    status, outs = _decode(GpuJpegDecoder("cuda"), [m[1:5] for m in mixed])
    for m, st, out in zip(mixed, status, outs):
        name, b, w, h = m[1:5]
        if m[0] == "good":
            assert st == 0 and np.array_equal(out, J.pillow_decode(b)), name
            continue
        expected = m[5]
        emu_status, emu_out = E.decode(b, w, h)
        assert st == emu_status, (name, int(st), emu_status)
        if expected is None:
            assert st == E.MALFORMED or (st == 0 and np.array_equal(out, J.pillow_decode(b))), name
        else:
            assert st == expected, (name, int(st))


def test_status_check_names_the_frame():
    good = J.pil_encode(J.content("video", 40, 30), "420", quality=80)
    status = GpuJpegDecoder("cuda").decode([good, good[:100]], [(40, 30)] * 2,
                                           [torch.empty((30, 40, 3), dtype=torch.uint8, device="cuda") for _ in range(2)])
    with pytest.raises(ValueError, match="frame 7: malformed"):
        GpuJpegDecoder.check(status, ["frame 6", "frame 7"])
    store = GpuVideoStore("cuda")
    with pytest.raises(ValueError, match="video 3 frame index 1"):
        store.put_jpeg(3, [good, J.pil_encode(J.content("video", 41, 30), "420", quality=80)])
    assert 3 not in store


def test_put_jpeg_equals_put_of_pillow_frames():
    frames = J.content("video", 171, 128)
    video = np.stack([np.roll(frames, 3 * k, axis=1) for k in range(12)])
    streams = [J.pil_encode(f, "420", quality=90) for f in video]
    store = GpuVideoStore("cuda")
    store.put_jpeg(0, streams)
    store.put(1, np.stack([J.pillow_decode(b) for b in streams]))
    assert torch.equal(store[0], store[1])
    assert store.bytes == 2 * video.size


def _dataset(variant):
    """Videos of different and odd sizes as JPEG frames, and a store of Pillow-decoded copies."""
    sizes = [(171, 128), (160, 121), (173, 131), (171, 128), (149, 113)]
    counts = [48, 61, 37, 52, 44]
    base = 1 if variant == "ucf" else 0
    enc = []
    store = GpuVideoStore("cuda")
    for i, ((w, h), n) in enumerate(zip(sizes, counts)):
        frames = J.content("video", w, h, i)
        video = [np.roll(np.roll(frames, 5 * k, axis=1), 2 * k, axis=0) for k in range(n)]
        enc.append([J.pil_encode(f, ("420", "422", "444")[i % 3], quality=85 + i) for f in video])
        store.put(i, np.stack([J.pillow_decode(b) for b in enc[i]]))

    def read_frames(video, frame_numbers):
        return [enc[video][f - base] for f in frame_numbers]
    return store, read_frames, counts


def _seed(s):
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)


@pytest.mark.parametrize("variant", ["ucf", "kinetics"])
@pytest.mark.parametrize("rank,world", [(0, 1), (1, 2)])
def test_jpeg_batches_equal_store_batches(variant, rank, world):
    store, read_frames, counts = _dataset(variant)
    kw = dict(batch_size=2, variant=variant, rank=rank, world=world, seed=3, drop_last=False)
    ref = PretrainBatches(store, counts, **kw)
    src = JpegPretrainBatches(read_frames, counts, **kw)
    n = 0
    for epoch in range(2):
        _seed(10 + epoch)
        want = [(x1.clone(), x2.clone(), tuple(l.clone() for l in lab)) for x1, x2, lab in ref(epoch)]
        _seed(10 + epoch)
        got = [(x1.clone(), x2.clone(), tuple(l.clone() for l in lab)) for x1, x2, lab in src(epoch)]
        assert len(got) == len(want) > 0
        for (a1, a2, la), (b1, b2, lb) in zip(got, want):
            assert torch.equal(a1, b1) and torch.equal(a2, b2)
            assert all(torch.equal(x, y) for x, y in zip(la, lb))
            n += 1
    assert n >= 4


def test_jpeg_batches_raise_at_the_next_request():
    store, read_frames, counts = _dataset("ucf")

    def broken(video, frame_numbers):
        out = read_frames(video, frame_numbers)
        return [b[:60] if video == 2 else b for b in out]
    src = JpegPretrainBatches(broken, counts, batch_size=1, variant="ucf", shuffle=False,
                              sizes=[tuple(store[i].shape[2:0:-1]) for i in range(len(counts))])
    it = src(0)
    next(it), next(it), next(it)                       # videos 0, 1, 2: the third batch holds the bad frames
    with pytest.raises(ValueError, match=r"video 2 frame \d+: malformed"):
        next(it)
