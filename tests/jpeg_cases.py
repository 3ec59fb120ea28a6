"""JPEG fixtures generated at test time (Pillow and cv2 encoders, byte-level rewrites) for the decoder tests.

good_cases() -> [(name, bytes, w, h)] that Pillow decodes and the decoder must reproduce byte for byte;
bad_cases()  -> [(name, bytes, w, h, expected status)] that it must reject (None: corrupt data libjpeg decodes without
                a warning; rejected, or decoded to Pillow's pixels).
"""
from __future__ import annotations

import io

import numpy as np
from PIL import Image

from cstp_b200.synthetic import synthetic_video
from tests.emulate_jpeg import MALFORMED, SIZE, UNSUPPORTED

SIZES = [(1, 1), (7, 5), (15, 17), (16, 16), (33, 47), (171, 128), (340, 256)]
SAMPLINGS = {"444": 0, "422": 1, "420": 2, "gray": None}
QUALITIES = [1, 50, 75, 95, 100]


def content(kind: str, w: int, h: int, seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed + 7 * w + h)
    if kind == "video":
        return synthetic_video(1, w, h, seed)[0]
    if kind == "noise":                                   # saturates IDCT outputs
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "flat":
        return np.broadcast_to(np.array([200, 30, 90], np.uint8), (h, w, 3)).copy()
    if kind == "edges":
        y, x = np.mgrid[0:h, 0:w]
        return np.stack([((x // 3) % 2) * 255, ((y // 5) % 2) * 255, (((x + y) // 4) % 2) * 255], -1).astype(np.uint8)
    raise ValueError(kind)


def pil_encode(img: np.ndarray, sampling: str, **kw) -> bytes:
    bio = io.BytesIO()
    if sampling == "gray":
        Image.fromarray(np.ascontiguousarray(img[:, :, 1])).save(bio, "JPEG", **kw)
    else:
        Image.fromarray(img).save(bio, "JPEG", subsampling=SAMPLINGS[sampling], **kw)
    return bio.getvalue()


def pillow_decode(b: bytes) -> np.ndarray:
    return np.asarray(Image.open(io.BytesIO(b)).convert("RGB"))


def segments(b: bytes):
    """[(marker, segment bytes including marker and length)] up to SOS, and the rest (SOS onwards)."""
    out, p = [], 2
    while True:
        m, seg = b[p + 1], (b[p + 2] << 8) | b[p + 3]
        if m == 0xDA:
            return out, b[p:]
        out.append((m, b[p:p + 2 + seg]))
        p += 2 + seg


def join(segs, rest) -> bytes:
    return b"\xff\xd8" + b"".join(s for _, s in segs) + rest


def split_tables(seg: bytes) -> list:
    """A DQT / DHT segment holding several tables -> one segment per table."""
    m, body, out, p = seg[1], seg[4:], [], 0
    while p < len(body):
        if m == 0xDB:
            n = 1 + 64 * ((body[p] >> 4) + 1)
        else:
            n = 17 + sum(body[p + 1:p + 17])
        t = body[p:p + n]
        out.append((m, bytes([0xFF, m]) + (len(t) + 2).to_bytes(2, "big") + t))
        p += n
    return out


def merge(segs, marker) -> list:
    body = b"".join(s[4:] for m, s in segs if m == marker)
    merged = (marker, bytes([0xFF, marker]) + (len(body) + 2).to_bytes(2, "big") + body)
    out, done = [], False
    for m, s in segs:
        if m == marker:
            if not done:
                out.append(merged)
                done = True
        else:
            out.append((m, s))
    return out


def rewrites(b: bytes) -> dict:
    """Byte-level variants of one baseline stream that decode to the same pixels."""
    segs, rest = segments(b)
    split = []
    for m, s in segs:
        split += split_tables(s) if m in (0xDB, 0xC4) else [(m, s)]
    tables = [x for x in split if x[0] in (0xDB, 0xC4)]
    others = [x for x in split if x[0] not in (0xDB, 0xC4)]
    app = (0xE5, b"\xff\xe5\x00\x08appx\x00\x01")
    com = (0xFE, b"\xff\xfe\x00\x07hello")
    out = {
        "split_tables": join(split, rest),
        "merged_tables": join(merge(merge(split, 0xDB), 0xC4), rest),
        "tables_after_sof": join(others + tables[::-1], rest),
        "app_com": join([app] + split[:2] + [com, app] + split[2:] + [com], rest),
        "fill_bytes": b"\xff\xd8" + b"".join(b"\xff\xff" + s for _, s in split) + b"\xff\xff" + rest,
    }
    # 16-bit quantisation tables with SOF1 (extended sequential)
    sixteen = []
    for m, s in split:
        if m == 0xDB:
            body = s[4:]
            t = bytes([0x10 | (body[0] & 15)]) + b"".join(int(v).to_bytes(2, "big") for v in body[1:65])
            sixteen.append((m, b"\xff\xdb" + (len(t) + 2).to_bytes(2, "big") + t))
        elif m == 0xC0:
            sixteen.append((0xC1, b"\xff\xc1" + s[2:]))
        else:
            sixteen.append((m, s))
    out["dqt16_sof1"] = join(sixteen, rest)
    return out


def good_cases(full: bool = True) -> list:
    cases = []
    for w, h in SIZES:
        big = w * h > 64 * 64
        for samp in SAMPLINGS:
            for q in QUALITIES:
                kinds = ("video", "noise", "flat", "edges")
                if big:          # the large sizes: every sampling, a spread of (quality, content) pairs
                    kinds = {1: ("edges",), 50: ("flat",), 75: ("video",), 95: ("video",), 100: ("noise",)}[q]
                for kind in kinds:
                    cases.append((f"{w}x{h}_{samp}_q{q}_{kind}", pil_encode(content(kind, w, h), samp, quality=q), w, h))
    img = content("video", 171, 128, 3)
    for samp in ("444", "422", "420", "gray"):
        for name, kw in (("optimize", dict(optimize=True)), ("rst_blocks1", dict(restart_marker_blocks=1)),
                         ("rst_blocks3", dict(restart_marker_blocks=3)), ("rst_rows1", dict(restart_marker_rows=1))):
            cases.append((f"171x128_{samp}_{name}", pil_encode(img, samp, quality=90, **kw), 171, 128))
    try:
        import cv2
    except ImportError:                                  # cv2 is optional: its cases are skipped without it
        cv2 = None
    if cv2 is not None:
        for w, h in ((171, 128), (33, 47), (340, 256)):
            im = content("video", w, h, 5)[:, :, ::-1].copy()
            for q in (60, 97):
                for tag, f in (("420", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420), ("422", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422),
                               ("444", cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444)):
                    ok, enc = cv2.imencode(".jpg", im, [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, f])
                    cases.append((f"cv2_{w}x{h}_{tag}_q{q}", enc.tobytes(), w, h))
            ok, enc = cv2.imencode(".jpg", np.ascontiguousarray(im[:, :, 0]), [cv2.IMWRITE_JPEG_QUALITY, 80])
            cases.append((f"cv2_{w}x{h}_gray", enc.tobytes(), w, h))
    for samp in ("420", "444", "gray"):
        base = pil_encode(content("video", 33, 47, 2), samp, quality=85)
        for name, b in rewrites(base).items():
            cases.append((f"rewrite_{samp}_{name}", b, 33, 47))
    if not full:
        cases = [c for c in cases if c[2] * c[3] <= 64 * 64 or c[0].startswith(("171x128", "cv2_171"))]
    return cases


def _set(b: bytes, pos: int, val: int) -> bytes:
    return b[:pos] + bytes([val]) + b[pos + 1:]


def bad_cases() -> list:
    img = content("video", 33, 47, 1)
    base = pil_encode(img, "420", quality=80)
    segs, rest = segments(base)
    sof = base.index(b"\xff\xc0")
    out = []
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", progressive=True)
    out.append(("progressive", b.getvalue(), 33, 47, UNSUPPORTED))
    b = io.BytesIO()
    Image.fromarray(img).convert("CMYK").save(b, "JPEG")
    out.append(("cmyk", b.getvalue(), 33, 47, UNSUPPORTED))
    try:
        import cv2
        ok, enc = cv2.imencode(".jpg", img, [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411])
        out.append(("cv2_411", enc.tobytes(), 33, 47, UNSUPPORTED))
    except ImportError:
        pass
    out.append(("precision12", _set(base, sof + 4, 12), 33, 47, UNSUPPORTED))
    out.append(("sof9", _set(base, sof + 1, 0xC9), 33, 47, UNSUPPORTED))
    out.append(("no_dht", join([s for s in segs if s[0] != 0xC4], rest), 33, 47, UNSUPPORTED))
    out.append(("no_dqt", join([s for s in segs if s[0] != 0xDB], rest), 33, 47, MALFORMED))
    # RGB: component ids 'R', 'G', 'B' without a JFIF segment; Adobe transform 0 likewise
    nojfif = [s for s in segs if s[0] != 0xE0]
    rgb = join(nojfif, rest)
    k = rgb.index(b"\xff\xc0") + 10
    for j, cid in enumerate((82, 71, 66)):
        rgb = _set(rgb, k + 3 * j, cid)
    sos = rgb.index(b"\xff\xda") + 5
    for j, cid in enumerate((82, 71, 66)):
        rgb = _set(rgb, sos + 2 * j, cid)
    out.append(("rgb_ids", rgb, 33, 47, UNSUPPORTED))
    adobe = (0xEE, b"\xff\xee\x00\x0eAdobe\x00\x64\x00\x00\x00\x00\x00")
    out.append(("adobe_transform0", join([adobe] + nojfif, rest), 33, 47, UNSUPPORTED))
    # a non-interleaved first scan (multi-scan baseline)
    ms = rest[:4] + bytes([1]) + rest[5:7] + rest[11:]
    ms = ms[:2] + (8).to_bytes(2, "big") + ms[4:]
    out.append(("multiscan", join(segs, ms), 33, 47, UNSUPPORTED))
    out.append(("size_w", base, 34, 47, SIZE))
    out.append(("size_h", base, 33, 46, SIZE))
    # truncation at every segment boundary and inside entropy data
    p, cuts = 2, [2]
    for _, s in segs:
        p += len(s)
        cuts.append(p)
    data0 = p + 2 + ((base[p + 2] << 8) | base[p + 3])      # first entropy-coded byte
    cuts += [p + 6, data0 + 20, data0 + (len(base) - data0) // 2, len(base) - 2, len(base) - 1]
    for c in cuts:
        out.append((f"truncated_{c}", base[:c], 33, 47, MALFORMED))
    # corrupt entropy data: a run of flipped bytes (kept clear of 0xFF so no marker is created) in a larger frame,
    # where the decoder cannot fall back into step before the data ends
    big = pil_encode(content("video", 171, 128, 1), "420", quality=80)
    segs, _ = segments(big)
    p = 2 + sum(len(s) for _, s in segs)
    data0 = p + 2 + ((big[p + 2] << 8) | big[p + 3])
    for start in (data0 + 8, data0 + (len(big) - data0) // 2, len(big) - 40):
        bb = bytearray(big)
        for j in range(start, start + 24):
            bb[j] = (bb[j] ^ 0x5A) if (bb[j] ^ 0x5A) != 0xFF else 0x00
        # Huffman codes resynchronise: libjpeg decodes these without a warning, so the decoder must either reject them
        # or return Pillow's pixels (expected status None)
        out.append((f"flipped_{start}", bytes(bb), 171, 128, None))
        ones = big[:start] + b"\xff\x00" * 12 + big[start + 24:]      # all-ones bits: no Huffman code matches
        out.append((f"bad_code_{start}", ones, 171, 128, MALFORMED))
    out.append(("extraneous_bytes", big[:-2] + b"\x12\x34\x56" + big[-2:], 171, 128, MALFORMED))
    return out
