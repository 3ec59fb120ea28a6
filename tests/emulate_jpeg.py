"""numpy stand-in of csrc/jpeg_decode.cu: the three stages of `cstp_jpeg_decode` with the kernels' integer arithmetic
and bounds logic, so that the decoder can be checked against Pillow on a machine without a GPU.

  parse()       stage A's marker walk (one lane per image in the kernel): validation, tables, the SOF / SOS fields.
  entropy()     stage A's entropy decode: one restart interval at a time, de-zigzagged int16 coefficients per block.
  idct()        stage B: dequantise + jpeg_idct_islow as libjpeg-turbo's SIMD code evaluates it (16-bit steps,
                saturation where jidctint.c's range-limit table would wrap).
  colour()      stage C: libjpeg's fancy upsampling (jdsample.c) with jdmainct.c's context rows, then jdcolor.c's
                YCbCr -> RGB tables.
  decode(b, w, h) -> (status, uint8 [h][w][3] or None).
"""
from __future__ import annotations

import numpy as np

OK, UNSUPPORTED, MALFORMED, SIZE = 0, 1, 2, 3

ZIGZAG = np.array([
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, 14, 21,
    28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61,
    54, 47, 55, 62, 63], dtype=np.int64)          # zigzag index -> natural (row-major) index


class _Reject(Exception):
    def __init__(self, code):
        self.code = code


def _u16(b, p):
    return (b[p] << 8) | b[p + 1]


class Huff:
    """A DHT table after jpeg_make_d_derived_tbl's checks: maxcode / valptr / mincode per code length."""

    def __init__(self, counts, vals, dc):
        if sum(counts) > 256:
            raise _Reject(MALFORMED)
        if dc and any(v > 15 for v in vals):
            raise _Reject(MALFORMED)
        self.vals = list(vals)
        self.maxcode = [-1] * 18
        self.mincode = [0] * 17
        self.valptr = [0] * 17
        code, k = 0, 0
        for l in range(1, 17):
            n = counts[l - 1]
            if n:
                self.valptr[l] = k
                self.mincode[l] = code
                code += n
                k += n
                if code > (1 << l):            # more codes of this length than the code space holds
                    raise _Reject(MALFORMED)
                self.maxcode[l] = code - 1
            code <<= 1
        self.maxcode[17] = 1 << 30


def parse(b: bytes, width: int, height: int) -> dict:
    """The marker walk up to the first SOS.  Raises _Reject with the status code."""
    n = len(b)
    if n < 4 or b[0] != 0xFF or b[1] != 0xD8:
        raise _Reject(MALFORMED)
    pos = 2
    qt = [None] * 4
    ht = {}
    sof = None
    dri = 0
    saw_jfif, adobe = False, -1
    while True:
        if pos >= n or b[pos] != 0xFF:
            raise _Reject(MALFORMED)
        while pos < n and b[pos] == 0xFF:          # fill bytes
            pos += 1
        if pos + 3 > n:
            raise _Reject(MALFORMED)
        m = b[pos]
        pos += 1
        if m in (0xC2, 0xC3, 0xC5, 0xC6, 0xC7, 0xC8, 0xC9, 0xCA, 0xCB, 0xCC, 0xCD, 0xCE, 0xCF, 0xDE, 0xDF):
            raise _Reject(UNSUPPORTED)               # progressive / lossless / hierarchical / arithmetic
        if not (m in (0xC0, 0xC1, 0xC4, 0xDA, 0xDB, 0xDD, 0xFE) or 0xE0 <= m <= 0xEF):
            raise _Reject(MALFORMED)                 # SOI, EOI, RSTn, DNL, TEM or an unknown marker before SOS
        seg = _u16(b, pos)
        end = pos + seg
        if seg < 2 or end > n:
            raise _Reject(MALFORMED)
        p = pos + 2
        if m in (0xC0, 0xC1):
            if sof is not None or seg < 8:
                raise _Reject(MALFORMED)
            if b[p] != 8:
                raise _Reject(UNSUPPORTED)
            h, w, nf = _u16(b, p + 1), _u16(b, p + 3), b[p + 5]
            if seg != 8 + 3 * nf or nf == 0:
                raise _Reject(MALFORMED)
            if nf not in (1, 3) or h == 0:
                raise _Reject(UNSUPPORTED)
            comps = []
            for c in range(nf):
                cid, hv, tq = b[p + 6 + 3 * c], b[p + 7 + 3 * c], b[p + 8 + 3 * c]
                hs, vs = hv >> 4, hv & 15
                if not (1 <= hs <= 4 and 1 <= vs <= 4) or tq > 3:
                    raise _Reject(MALFORMED)
                comps.append((cid, hs, vs, tq))
            if w == 0:
                raise _Reject(MALFORMED)
            if (w, h) != (width, height):
                raise _Reject(SIZE)
            if nf == 3:
                if comps[0][1:3] not in ((1, 1), (2, 1), (2, 2)) or comps[1][1:3] != (1, 1) or comps[2][1:3] != (1, 1):
                    raise _Reject(UNSUPPORTED)
            sof = comps
        elif m == 0xC4:
            while p < end:
                tc, th = b[p] >> 4, b[p] & 15
                if tc > 1 or th > 3 or p + 17 > end:
                    raise _Reject(MALFORMED)
                counts = list(b[p + 1:p + 17])
                tot = sum(counts)
                if p + 17 + tot > end:
                    raise _Reject(MALFORMED)
                ht[(tc, th)] = Huff(counts, b[p + 17:p + 17 + tot], tc == 0)
                p += 17 + tot
        elif m == 0xDB:
            while p < end:
                pq, tq = b[p] >> 4, b[p] & 15
                if pq > 1 or tq > 3 or p + 1 + 64 * (pq + 1) > end:
                    raise _Reject(MALFORMED)
                q = np.zeros(64, dtype=np.int64)
                for k in range(64):
                    q[ZIGZAG[k]] = _u16(b, p + 1 + 2 * k) if pq else b[p + 1 + k]
                qt[tq] = q
                p += 1 + 64 * (pq + 1)
        elif m == 0xDD:
            if seg != 4:
                raise _Reject(MALFORMED)
            dri = _u16(b, p)
        elif m == 0xE0:
            if seg - 2 >= 14 and bytes(b[p:p + 5]) == b"JFIF\0":
                saw_jfif = True
        elif m == 0xEE:
            if seg - 2 >= 12 and bytes(b[p:p + 5]) == b"Adobe":
                adobe = b[p + 11]
        elif m == 0xDA:
            if sof is None or seg < 3:
                raise _Reject(MALFORMED)
            ns = b[p]
            if seg != 6 + 2 * ns:
                raise _Reject(MALFORMED)
            if ns != len(sof):
                raise _Reject(UNSUPPORTED)              # one interleaved scan only
            tabs = []
            for c in range(ns):
                cs, t = b[p + 1 + 2 * c], b[p + 2 + 2 * c]
                if cs != sof[c][0]:
                    raise _Reject(UNSUPPORTED)
                if (t >> 4) > 3 or (t & 15) > 3:
                    raise _Reject(MALFORMED)
                tabs.append((t >> 4, t & 15))
            q = p + 1 + 2 * ns
            if b[q] != 0 or b[q + 1] != 63 or b[q + 2] != 0:
                raise _Reject(UNSUPPORTED)
            for c in range(ns):
                if qt[sof[c][3]] is None:
                    raise _Reject(MALFORMED)
                if (0, tabs[c][0]) not in ht or (1, tabs[c][1]) not in ht:
                    raise _Reject(UNSUPPORTED)          # libjpeg-turbo would substitute the standard tables
            if ns == 3 and not saw_jfif and (adobe == 0 or (adobe < 0 and [c[0] for c in sof] == [82, 71, 66])):
                raise _Reject(UNSUPPORTED)              # RGB, not YCbCr
            if ns == 1:
                comps = [(sof[0][0], 1, 1, sof[0][3])]
            else:
                comps = sof
            return dict(comps=comps, qt=[qt[c[3]] for c in comps], dc=[ht[(0, t[0])] for t in tabs],
                        ac=[ht[(1, t[1])] for t in tabs], dri=dri, data=end)
        pos = end


def layout(comps, width, height):
    """Padded MCU-grid geometry of the coefficient / plane layout every stage shares."""
    hmax = max(c[1] for c in comps)
    vmax = max(c[2] for c in comps)
    mcux = -(-width // (8 * hmax))
    mcuy = -(-height // (8 * vmax))
    geo = []
    for _, hs, vs, _ in comps:
        geo.append(dict(bw=mcux * hs, bh=mcuy * vs, dw=-(-width * hs // hmax), dh=-(-height * vs // vmax), hs=hs, vs=vs))
    return hmax, vmax, mcux, mcuy, geo


def intervals(b: bytes, start: int, n_int: int):
    """Restart intervals of the entropy-coded data: [(begin, end)], `end` before the fill bytes of the marker that closes
    it.  The data must close with RST0, RST1, ... between intervals and EOI after the last."""
    n = len(b)
    out = []
    p = begin = start
    while True:
        while p + 1 < n and not (b[p] == 0xFF and b[p + 1] not in (0x00, 0xFF)):
            p += 1
        if p + 1 >= n:
            raise _Reject(MALFORMED)                    # truncated: no closing marker
        m = b[p + 1]
        e = p
        while e > begin and b[e - 1] == 0xFF:
            e -= 1
        k = len(out)
        out.append((begin, e))
        if m == 0xD9:
            if k != n_int - 1:
                raise _Reject(MALFORMED)
            return out
        if m != 0xD0 + (k & 7) or k >= n_int - 1:
            raise _Reject(MALFORMED)
        p += 2
        begin = p


class _Bits:
    def __init__(self, b, begin, end):
        self.b, self.pos, self.end = b, begin, end
        self.acc, self.n, self.fake = 0, 0, 0

    def fill(self):
        while self.n <= 56:
            if self.pos < self.end:
                v = self.b[self.pos]
                self.pos += 2 if v == 0xFF else 1          # FF 00 stuffing (every FF inside an interval is stuffed)
            else:
                v = 0
                self.fake += 1
            self.acc |= v << (56 - self.n)
            self.n += 8

    def get(self, k):
        v = self.acc >> (64 - k)
        self.acc = (self.acc << k) & 0xFFFFFFFFFFFFFFFF
        self.n -= k
        return v

    def sym(self, t: Huff):
        for l in range(1, 17):
            code = self.acc >> (64 - l)
            if code <= t.maxcode[l]:
                self.get(l)
                return t.vals[t.valptr[l] + code - t.mincode[l]]
        raise _Reject(MALFORMED)


def _extend(v, s):
    return v - (1 << s) + 1 if v < (1 << (s - 1)) else v


def entropy(b: bytes, hdr: dict, width: int, height: int):
    comps = hdr["comps"]
    _, _, mcux, mcuy, geo = layout(comps, width, height)
    coef = [np.zeros((g["bh"], g["bw"], 64), dtype=np.int16) for g in geo]
    total = mcux * mcuy
    ri = hdr["dri"] or total
    n_int = -(-total // ri)
    for k, (begin, end) in enumerate(intervals(b, hdr["data"], n_int)):
        bits = _Bits(b, begin, end)
        pred = [0] * len(comps)
        for m in range(k * ri, min(total, (k + 1) * ri)):
            my, mx = divmod(m, mcux)
            for c, (_, hs, vs, _) in enumerate(comps):
                for by in range(vs):
                    for bx in range(hs):
                        blk = coef[c][my * vs + by, mx * hs + bx]
                        bits.fill()
                        s = bits.sym(hdr["dc"][c])
                        if s:
                            bits.fill()
                            pred[c] += _extend(bits.get(s), s)
                        blk[0] = np.int16(np.int32(pred[c]).astype(np.int16))
                        z = 1
                        while z < 64:
                            bits.fill()
                            rs = bits.sym(hdr["ac"][c])
                            r, s = rs >> 4, rs & 15
                            if s:
                                z += r
                                if z > 63:
                                    raise _Reject(MALFORMED)
                                blk[ZIGZAG[z]] = _extend(bits.get(s), s)
                            elif r == 15:
                                z += 15
                            else:
                                break
                            z += 1
        if bits.n < 8 * bits.fake or bits.pos < bits.end or bits.n - 8 * bits.fake >= 8:
            raise _Reject(MALFORMED)                    # ran past the interval's data, or left whole bytes unread
    return coef


F = dict(c0_298=2446, c0_390=3196, c0_541=4433, c0_765=6270, c0_899=7373, c1_175=9633, c1_501=12299, c1_847=15137,
         c1_961=16069, c2_053=16819, c2_562=20995, c3_072=25172)


def _s16(x):
    return ((x + 32768) & 0xFFFF) - 32768


def _idct_1d(x0, x1, x2, x3, x4, x5, x6, x7):
    """One pass of jpeg_idct_islow on int16-valued int32 arrays, as libjpeg-turbo's SIMD islow kernels evaluate it (the
    ones Pillow's libjpeg-turbo runs): the products of the rotations are exact in 32 bits, but the sums x0 +- x4,
    x7 + x3 and x5 + x1 are formed in 16 bits first.  Returns the 8 outputs before descaling."""
    t3 = x2 * (F["c0_541"] + F["c0_765"]) + x6 * F["c0_541"]
    t2 = x2 * F["c0_541"] + x6 * (F["c0_541"] - F["c1_847"])
    t0 = _s16(x0 + x4) << 13
    t1 = _s16(x0 - x4) << 13
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    z3 = _s16(x7 + x3)
    z4 = _s16(x5 + x1)
    z3, z4 = z3 * (F["c1_175"] - F["c1_961"]) + z4 * F["c1_175"], z3 * F["c1_175"] + z4 * (F["c1_175"] - F["c0_390"])
    o0 = x7 * (F["c0_298"] - F["c0_899"]) + x1 * -F["c0_899"] + z3
    o1 = x5 * (F["c2_053"] - F["c2_562"]) + x3 * -F["c2_562"] + z4
    o2 = x5 * -F["c2_562"] + x3 * (F["c3_072"] - F["c2_562"]) + z3
    o3 = x7 * -F["c0_899"] + x1 * (F["c1_501"] - F["c0_899"]) + z4
    return [t10 + o3, t11 + o2, t12 + o1, t13 + o0, t13 - o0, t12 - o1, t11 - o2, t10 - o3]


def idct(coef: np.ndarray, q: np.ndarray) -> np.ndarray:
    """int16 [bh][bw][64] natural-order coefficients, quant table (natural order) -> uint8 plane [bh*8][bw*8].

    libjpeg-turbo's SIMD jpeg_idct_islow: the dequantised coefficient is the low 16 bits of coef * q, each pass's
    descaled output saturates to int16, and the last one to [-128, 127] before the +128 level shift -- a clamp where
    the C code's range-limit table (`& RANGE_MASK`) would wrap.  Valid streams never reach either limit."""
    bh, bw = coef.shape[:2]
    c = _s16(coef.astype(np.int32) * q.astype(np.int32)).reshape(bh, bw, 8, 8)   # [.., row u, col v]
    cols = _idct_1d(*[c[:, :, u, :] for u in range(8)])                          # pass 1: down each column
    ws = np.stack([np.clip((t + (1 << 10)) >> 11, -32768, 32767) for t in cols], axis=2)   # [.., y, col]
    rows = _idct_1d(*[ws[:, :, :, v] for v in range(8)])                           # pass 2: along each row
    out = np.stack([np.clip((t + (1 << 17)) >> 18, -128, 127) + 128 for t in rows], axis=3)   # [.., y, x]
    return out.astype(np.uint8).transpose(0, 2, 1, 3).reshape(bh * 8, bw * 8)


def _fancy(plane, g, width, height, hmax, vmax):
    """A chroma plane upsampled to width x height (int32), as jdsample.c does for its factor."""
    dw, dh = g["dw"], g["dh"]
    hs_up, vs_up = hmax // g["hs"], vmax // g["vs"]
    p = plane[:dh, :dw].astype(np.int32)
    ys, xs = np.arange(height), np.arange(width)
    if hs_up == 1 and vs_up == 1:
        return p[:height, :width]
    if dw <= 2:                                        # jinit_upsampler: no fancy upsampling this narrow
        return p[ys // vs_up][:, xs // hs_up]
    j = xs // 2
    left = (xs & 1) == 0
    nb = np.where(left, np.maximum(j - 1, 0), np.minimum(j + 1, dw - 1))
    if vs_up == 1:                                     # h2v1_fancy_upsample
        return (3 * p[:, j] + p[:, nb] + np.where(left, 1, 2)) >> 2
    i = ys // 2
    vn = np.where((ys & 1) == 0, np.maximum(i - 1, 0), np.minimum(i + 1, dh - 1))
    cs = 3 * p[i] + p[vn]                              # h2v2_fancy_upsample: column sums, then across
    return (3 * cs[:, j] + cs[:, nb] + np.where(left, 8, 7)) >> 4


ONE_HALF = 1 << 15


def colour(planes, hdr, width, height) -> np.ndarray:
    comps = hdr["comps"]
    hmax, vmax, _, _, geo = layout(comps, width, height)
    y = planes[0][:height, :width].astype(np.int32)
    if len(comps) == 1:
        return np.repeat(y[:, :, None], 3, axis=2).astype(np.uint8)
    cb = _fancy(planes[1], geo[1], width, height, hmax, vmax) - 128
    cr = _fancy(planes[2], geo[2], width, height, hmax, vmax) - 128
    r = y + ((91881 * cr + ONE_HALF) >> 16)
    g = y + ((-22554 * cb + ONE_HALF - 46802 * cr) >> 16)
    b = y + ((116130 * cb + ONE_HALF) >> 16)
    return np.clip(np.stack([r, g, b], -1), 0, 255).astype(np.uint8)


def decode(b: bytes, width: int, height: int):
    """-> (status, uint8 [height][width][3] or None)."""
    b = memoryview(bytes(b))
    try:
        hdr = parse(b, width, height)
        coef = entropy(b, hdr, width, height)
    except _Reject as r:
        return r.code, None
    planes = [idct(c, q) for c, q in zip(coef, hdr["qt"])]
    return OK, colour(planes, hdr, width, height)
