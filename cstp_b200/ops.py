"""Host-side operator layer over the C ABI: builds implicit-GEMM plans (TMA views, tap lists, tile boxes) for the
forward / dgrad / wgrad of the factorised R(2+1)D convolutions and linear layers, and wraps the elementwise,
loss and optimiser kernels.  torch is used only for device memory and streams.

Layout conventions: activations are bf16 (N, T, H, W, Cp) with Cp = channels padded to a multiple of 16;
packed forward weights are bf16 [Np][taps*Kc] with Kc = Cp_in rounded up to 64.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from itertools import product

import torch

from . import lib as L


def pad16(c: int) -> int:
    return (c + 15) // 16 * 16


def pad64(c: int) -> int:
    return (c + 63) // 64 * 64


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _require_cuda(*tensors) -> None:
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise L.CstpError("cstp_b200 ops need CUDA tensors: there is no CPU fallback")


def require_device(*tensors) -> None:
    """Public guard used by the module layer: the product path only accepts CUDA tensors."""
    _require_cuda(*tensors)


# ------------------------------------------------------------------------------------------------ geometry
def pick_box(W: int, H: int, T: int, N: int, rows: int) -> tuple[int, int, int, int]:
    """Chooses the (bw, bh, bt, bn) box with bw*bh*bt*bn == rows that wastes the fewest positions."""
    best = None
    divs = [d for d in (1, 2, 4, 8, 16, 32, 64, 128) if d <= rows]
    for bw in divs:
        for bh in divs:
            if bw * bh > rows:
                continue
            for bt in divs:
                if bw * bh * bt > rows:
                    continue
                bn = rows // (bw * bh * bt)
                if bw * bh * bt * bn != rows or bn > 256:
                    continue
                tiles = math.ceil(W / bw) * math.ceil(H / bh) * math.ceil(T / bt) * math.ceil(N / bn)
                # tie-break: prefer wide inner boxes (fewer, longer TMA rows), then small bn
                key = (tiles, -bw, -bh, bn)
                if best is None or key < best[0]:
                    best = (key, (bw, bh, bt, bn))
    return best[1]


def view5_geometry(shape, parity=(0, 0, 0), stride=(1, 1, 1)):
    """(element offset, dims (C,W,H,T,N), element strides of W,H,T,N) of the stride-parity sub-lattice of an
    (N, T, H, W, Cp) tensor.  Pure shape arithmetic (also interpreted by the CPU emulator in tests/)."""
    N, T, H, W, Cp = shape
    (rt, rh, rw), (st, sh, sw) = parity, stride
    off = ((rt * H + rh) * W + rw) * Cp
    dims = (Cp, (W - rw + sw - 1) // sw, (H - rh + sh - 1) // sh, (T - rt + st - 1) // st, N)
    strides = (sw * Cp, sh * W * Cp, st * H * W * Cp, T * H * W * Cp)
    return off, dims, strides


def _view5(x: torch.Tensor, parity=(0, 0, 0), stride=(1, 1, 1)) -> L.Tensor5:
    """TMA view (C, W, H, T, N) of the stride-parity sub-lattice of an (N, T, H, W, Cp) bf16 tensor."""
    off, dims, strides = view5_geometry(tuple(x.shape), parity, stride)
    t5 = L.Tensor5()
    es = x.element_size()
    t5.ptr = x.data_ptr() + off * es
    for i, d in enumerate(dims):
        t5.dims[i] = d
    for i, s_ in enumerate(strides):
        t5.strides[i] = s_ * es
    return t5


@dataclass
class ConvGeom:
    kernel: tuple[int, int, int]
    stride: tuple[int, int, int] = (1, 1, 1)
    pad: tuple[int, int, int] = (0, 0, 0)
    pad_hi: tuple[int, int, int] | None = None     # padding at the far end of every axis when it differs from `pad`

    @property
    def taps(self) -> int:
        return self.kernel[0] * self.kernel[1] * self.kernel[2]

    def out_dims(self, T: int, H: int, W: int) -> tuple[int, int, int]:
        (kt, kh, kw), (st, sh, sw), (pt, ph, pw) = self.kernel, self.stride, self.pad
        qt, qh, qw = self.pad_hi or self.pad
        return ((T + pt + qt - kt) // st + 1, (H + ph + qh - kh) // sh + 1, (W + pw + qw - kw) // sw + 1)


def fwd_taps(g: ConvGeom):
    """Per tap (kt,kh,kw raster order): the stride-parity class it reads and the integer offset d such that
    in = stride*(out + d) + parity.  Returns (parities, [(map_id, dw, dh, dt, tap_index)])."""
    maps, taps = [], []
    (kt, kh, kw), (st, sh, sw), (pt, ph, pw) = g.kernel, g.stride, g.pad
    ti = 0
    for a in range(kt):
        for b in range(kh):
            for c in range(kw):
                q = (a - pt, b - ph, c - pw)
                r = (q[0] % st, q[1] % sh, q[2] % sw)
                d = ((q[0] - r[0]) // st, (q[1] - r[1]) // sh, (q[2] - r[2]) // sw)
                if r not in maps:
                    maps.append(r)
                taps.append((maps.index(r), d[2], d[1], d[0], ti))
                ti += 1
    if len(maps) > L.CSTP_MAX_AMAPS:
        raise L.CstpError("too many stride-parity views for one convolution")
    return maps, taps


def dgrad_classes(shape_dx, geom: ConvGeom):
    """Stride-parity classes of dx for the transposed convolution.  For class c, dx[s*a + c] sums the taps k with
    (c + p - k) % s == 0 read at g[a + (c + p - k)/s].  Yields dicts with taps (dw,dh,dt,tap_index), the tile space,
    the element offset/strides of the class inside dx; classes without taps have taps == []."""
    N, T, H, W, Ci = shape_dx
    (kt, kh, kw), (st, sh, sw), (pt, ph, pw) = geom.kernel, geom.stride, geom.pad
    out = []
    for ct, ch, cw in product(range(st), range(sh), range(sw)):
        taps = []
        ti = 0
        for a in range(kt):
            for b in range(kh):
                for c in range(kw):
                    e = (ct + pt - a, ch + ph - b, cw + pw - c)
                    if e[0] % st == 0 and e[1] % sh == 0 and e[2] % sw == 0:
                        taps.append((e[2] // sw, e[1] // sh, e[0] // st, ti))
                    ti += 1
        space = ((W - cw + sw - 1) // sw, (H - ch + sh - 1) // sh, (T - ct + st - 1) // st, N)
        if min(space) <= 0:
            continue
        out.append(dict(cls=(ct, ch, cw), taps=taps, space=space, off=((ct * H + ch) * W + cw) * Ci,
                        ostrides=(sw * Ci, sh * W * Ci, st * H * W * Ci, T * H * W * Ci)))
    return out


def _fwd_taps(x: torch.Tensor, g: ConvGeom):
    """TMA views + taps of a convolution over x.  A stride-parity class can be EMPTY (e.g. T = 1 under a stride-2
    temporal conv has no odd frames): its taps only ever read padding, so they are redirected to view 0 at an offset far
    outside the tensor, where TMA zero-fills -- the tap list (and the weight-gradient chunk layout) keeps its shape."""
    maps, taps = fwd_taps(g)
    geo = [view5_geometry(tuple(x.shape), r, g.stride) for r in maps]
    alive = [i for i, (_, dims, _) in enumerate(geo) if min(dims) > 0]
    if len(alive) == len(maps):
        return [_view5(x, r, g.stride) for r in maps], taps
    remap = {old: new for new, old in enumerate(alive)}
    far = 1 << 20
    taps = [(remap[m], dw, dh, dt, ti) if m in remap else (0, far, far, far, ti) for (m, dw, dh, dt, ti) in taps]
    return [_view5(x, maps[i], g.stride) for i in alive], taps


class _Plan:
    """Owns a C plan handle plus references to every tensor whose address the plan baked in."""

    def __init__(self, handle, destroy, keep):
        self.handle, self._destroy, self._keep = handle, destroy, keep

    def __del__(self):
        try:
            if self.handle:
                self._destroy(self.handle)
        except Exception:
            pass


class ConvPlan(_Plan):
    def run(self):
        L.check(L.load().cstp_conv_plan_run(self.handle, _stream()))

    @property
    def cluster(self) -> int:
        """CTAs per cluster of the launch (2: CTA pairs with multicast weight tiles)."""
        return int(L.load().cstp_conv_plan_cluster(self.handle))


class WgradPlan(_Plan):
    splits: int = 1

    def run(self):
        L.check(L.load().cstp_wgrad_plan_run(self.handle, _stream()))


def _default_n_tile(Np: int) -> int:
    if Np <= 256:
        return Np
    # fewest tiles, each a multiple of 16 and <= 256, as even as possible
    nt = math.ceil(Np / 256)
    return pad16(math.ceil(Np / nt))


def _set_prologue(d, prologue: "BNState | None", a_channels: int) -> tuple:
    """Fills desc.pro from the BatchNorm state of the unit that PRODUCED the operand (its raw output is what the kernel
    reads); returns the tensors the plan must keep alive."""
    if prologue is None:
        return ()
    if prologue.Cp != a_channels:
        raise L.CstpError(f"prologue BatchNorm has {prologue.Cp} padded channels, the operand {a_channels}")
    d.pro.scale, d.pro.shift = prologue.scale.data_ptr(), prologue.shift.data_ptr()
    d.pro.groups, d.pro.Cp = prologue.groups, prologue.Cp
    return (prologue.scale, prologue.shift)


def _make_conv_plan(views, taps, a_channels, w_packed, Np, tile_space, box, out, out_f32, out_off, ostrides, bias,
                    accumulate, n_tile, keep, prologue=None, classes=None) -> ConvPlan:
    """classes: [(first tap, number of taps, output element offset)] -- several tap classes with the same tile space run
    as one launch (the stride-parity classes of a strided dgrad)."""
    lib = L.load()
    d = L.ConvDesc()
    if classes and len(classes) > 1:
        d.n_classes = len(classes)
        for i, (t0, nt, off) in enumerate(classes):
            d.cls_first_tap[i], d.cls_n_taps[i], d.cls_out_off[i] = t0, nt, off
    keep = keep + _set_prologue(d, prologue, a_channels)
    d.n_amaps = len(views)
    for i, v in enumerate(views):
        d.amap[i] = v
    d.a_channels = a_channels
    d.n_taps = len(taps)
    for i, (mid, dw, dh, dt, koff) in enumerate(taps):
        d.taps[i] = L.Tap(mid, dw, dh, dt, koff)
    d.w_packed = w_packed.data_ptr()
    d.Np = Np
    d.Ktot = w_packed.shape[1]
    d.n_tile = n_tile or _default_n_tile(Np)
    d.Wt, d.Ht, d.Tt, d.Nt = tile_space
    d.bw, d.bh, d.bt, d.bn = box
    d.out_bf16 = 0 if out is None else out.data_ptr()
    d.out_f32 = 0 if out_f32 is None else out_f32.data_ptr()
    d.out_off = out_off
    d.osw, d.osh, d.ost, d.osn = ostrides
    d.bias = 0 if bias is None else bias.data_ptr()
    d.accumulate = int(accumulate)
    h = C.c_void_p()
    L.check(lib.cstp_conv_plan_create(C.byref(d), C.byref(h)))
    return ConvPlan(h, lib.cstp_conv_plan_destroy, keep)


class ConvHaloPlan(_Plan):
    resident: bool = False
    stat_blocks: int = 0         # > 0: the kernel also writes BatchNorm statistics partials (that many blocks)

    def run(self):
        L.check(L.load().cstp_conv_halo_plan_run(self.handle, _stream()))


# same budget as csrc/common.h kSmemBudget
SMEM_LIMIT = 227 * 1024
SMEM_BUDGET = SMEM_LIMIT - 1024 - 256


def conv_halo_layout(tile_space, taps, a_channels: int, Np: int):
    """The 2-D halo layout when it applies and keeps the full-width weights resident, else the one-axis halo layout."""
    lay = _conv_halo_layout(tile_space, taps, a_channels, Np, True)
    if lay is not None and lay["pitch"] != 8 and lay["resident"] and lay["n_tile"] == min(Np, 256):
        return lay
    return _conv_halo_layout(tile_space, taps, a_channels, Np, False)


def _conv_halo_layout(tile_space, taps, a_channels: int, Np: int, halo_2d: bool):
    """Geometry of csrc/conv_halo.cu for a single-view (stride-1) tap list [(dw, dh, dt, k_off)], or None when the
    layer does not qualify (then csrc/conv_gemm.cu is used).  Pure shape arithmetic.

    The taps must vary along t only (3x1x1: one load group, halo along t) or along h and w only (1x3x3: one load group
    per dw, halo along h).  Returns dict(box, halo, groups [(dw, dh, dt, first_tap, n_taps)], taps [(a_shift, k_off)]
    in group order, n_tile, a_bytes, resident)."""
    Wt, Ht, Tt, Nt = tile_space
    if len(taps) < 2 or len(taps) > 16:
        return None
    dws, dhs, dts = sorted({t[0] for t in taps}), sorted({t[1] for t in taps}), sorted({t[2] for t in taps})
    temporal = len(dws) == 1 and len(dhs) == 1 and len(dts) > 1
    spatial = len(dts) == 1 and len(dhs) > 1
    if not (temporal or spatial) or len(dws) > 4:
        return None
    if temporal and (dws[0] != 0 or dhs[0] != 0):
        return None
    span = (dts[-1] - dts[0]) if temporal else (dhs[-1] - dhs[0])
    best = None
    for bw in (4, 8, 16, 32, 64, 128):
        for bh in (1, 2, 4, 8, 16, 32):
            for bt in ((1, 2, 4, 8, 16, 32) if temporal else (1,)):
                if bw * bh * bt != 128:
                    continue
                unit = bw * bh if temporal else bw          # rows per step of the halo axis
                if unit % 8:
                    continue
                tiles = math.ceil(Wt / bw) * math.ceil(Ht / bh) * math.ceil(Tt / bt)
                rows = (bw * bh * (bt + span)) if temporal else (bw * (bh + span))
                key = (tiles, tiles * rows * (1 if temporal else len(dws)), -bw)
                if best is None or key < best[0]:
                    best = (key, (bw, bh, bt, 1), rows, unit)
    if best is None:
        return None
    _, box, rows, unit = best
    halo = (0, 0, span) if temporal else (0, span, 0)
    groups, out_taps = [], []
    pitch = 8
    # 1 x k x k filters, 2-D halo: ONE staged box (8 + wspan) x (16 + span) serves every tap.  A tap's 128 rows are then
    # 16 runs of 8 consecutive box rows (one swizzle atom each) spaced by the box width: atom pitch 8 + wspan rows,
    # a_shift in whole rows.  Taken when it does not need more tiles than the best one-axis layout (56 x 56 planes: 28
    # tiles either way, 180 staged rows per 64-channel chunk instead of 3 x 160).
    wspan = dws[-1] - dws[0]
    if (halo_2d and spatial and len(dws) > 1 and dws == list(range(dws[0], dws[-1] + 1))
            and math.ceil(Wt / 8) * math.ceil(Ht / 16) * Tt <= best[0][0]):
        box, halo, pitch = (8, 16, 1, 1), (wspan, span, 0), 8 + wspan
        rows = (8 + wspan) * (16 + span)
        groups.append((dws[0], dhs[0], dts[0], 0, len(taps)))
        # same accumulation order as the one-axis layout (dw outermost): single-chunk layers keep their bits
        for (dw, dh, dt, k_off) in sorted(taps, key=lambda t: (t[0], t[1])):
            out_taps.append((((dh - dhs[0]) * pitch + (dw - dws[0])) * 128, k_off))
    elif temporal:
        groups.append((0, 0, dts[0], 0, len(taps)))
        for (dw, dh, dt, k_off) in sorted(taps, key=lambda t: t[2]):
            out_taps.append(((dt - dts[0]) * unit * 128, k_off))
    else:
        for dw in dws:
            mine = sorted([t for t in taps if t[0] == dw], key=lambda t: t[1])
            groups.append((dw, dhs[0], dts[0], len(out_taps), len(mine)))
            for (_, dh, _, k_off) in mine:
                out_taps.append(((dh - dhs[0]) * unit * 128, k_off))
    a_bytes = (rows * 128 + 1023) // 1024 * 1024          # stage pitch (csrc/conv_halo.cu a_stride)
    chunks = pad64(a_channels) // 64
    # a channel tail of exactly 16 / 32 beyond a multiple of 64 is staged with 32 / 64-byte rows (csrc/conv_halo.cu)
    tail = a_channels % 64 if (a_channels > 64 and a_channels % 64 in (16, 32)) else 0
    k_bytes_per_row = ((chunks - 1) * 128 + tail * 2) if tail else chunks * 128      # resident weight bytes per (tap, n)
    # N tile: keep all weight K-blocks resident when they fit beside 3 activation stages, splitting N in two if needed
    n_tile, resident = (Np if Np <= 256 else _default_n_tile(Np)), False
    for cand in ([Np] if Np <= 256 else []) + ([pad16(math.ceil(Np / 2))] if Np > 64 else []):
        # (a 2-D halo stage feeds every tap of the filter: two of them already double-buffer whole K-blocks)
        if cand <= 256 and len(taps) * k_bytes_per_row * cand + (3 if pitch == 8 else 2) * a_bytes <= SMEM_BUDGET:
            n_tile, resident = cand, True
            break
    if not resident:
        per_stage = a_bytes + max(g[4] for g in groups) * n_tile * 128
        if 2 * per_stage > SMEM_BUDGET:
            return None
    return dict(box=box, halo=halo, groups=groups, taps=out_taps, n_tile=n_tile, a_bytes=a_bytes, resident=resident,
                tail=tail, pitch=pitch)


def slab_tables(G: int, nslots: int, Np: int):
    """The per-input-slab tables of csrc/conv_halo.cu's slab mode, in issue order: [(input slab s, overwrite?, first
    accumulator column, first row of the stacked weight block, MMA width)] -- restated here for the CPU layout
    interpreter (tests/test_geometry.py); cstp_conv_halo_plan_create derives the same."""
    span, n_in = nslots - 1, G + nslots - 1
    order, covered = [], 0
    while covered < G:
        s = min(covered + span, n_in - 1)
        order.append(s)
        covered = min(s, G - 1) + 1
    n_init = len(order)
    order += [s for s in range(n_in) if s not in order]
    out = []
    for i, s in enumerate(order):
        o_lo, o_hi = max(0, s - span), min(G - 1, s)
        out.append((s, i < n_init, o_lo * Np, (span - s + o_lo) * Np, (o_hi - o_lo + 1) * Np))
    return out


def conv_slab_layout(tile_space, taps, a_channels: int, Np: int, G: int = 4):
    """Slab-mode geometry of csrc/conv_halo.cu (include/cstp_b200.h cstp_halo_slabs) for a stride-1 1 x k x k tap list
    [(dw, dh, dt, k_off)] of a layer with Np == 64 output columns, or None: G output rows per tile (slab axis h), every
    input row staged as ONE box with a halo along w (the w taps are row shifts of it).  Same dict as conv_halo_layout plus
    `slabs` = (G, 1, nslots); taps are listed w tap by w tap, the h taps in DEscending offset order."""
    Wt, Ht, Tt, Nt = tile_space
    if Np != 64 or G < 2 or G * Np > 256 or len(taps) < 2 or len(taps) > 16:
        return None
    dws, dhs, dts = sorted({t[0] for t in taps}), sorted({t[1] for t in taps}), sorted({t[2] for t in taps})
    consecutive = lambda v: v == list(range(v[0], v[-1] + 1))      # noqa: E731
    if not (len(dts) == 1 and len(dhs) > 1 and consecutive(dws) and consecutive(dhs) and len(taps) == len(dws) * len(dhs)):
        return None
    wspan = dws[-1] - dws[0]
    nslots = len(dhs)
    if nslots > 4 or nslots * Np > 256 or Ht < G:
        return None
    # 128 positions with extent 1 along h, 8 along w (one swizzle atom per run when the box has a w halo)
    best = None
    for bt in (16, 8, 4, 2, 1):                  # extent along t, the rest along n
        bn = 16 // bt
        key = (math.ceil(Tt / bt) * math.ceil(Nt / bn), bn)
        if best is None or key < best[0]:
            best = (key, bt, bn)
    _, bt, bn = best
    box = (8, 1, bt, bn)
    rows = (8 + wspan) * bt * bn
    pitch = 8 + wspan if wspan else 8
    a_bytes = (rows * 128 + 1023) // 1024 * 1024
    chunks = pad64(a_channels) // 64
    tail = a_channels % 64 if (a_channels > 64 and a_channels % 64 in (16, 32)) else 0
    k_bytes_per_row = ((chunks - 1) * 128 + tail * 2) if tail else chunks * 128
    if len(taps) * k_bytes_per_row * Np + 2 * a_bytes > SMEM_BUDGET:
        return None
    by_off = {(t[0], t[1], t[2]): t[3] for t in taps}
    out_taps = [((dw - dws[0]) * 128, by_off[(dw, dh, dts[0])]) for dw in dws for dh in reversed(dhs)]
    groups = [(dws[0], dhs[0], dts[0], 0, len(taps))]
    return dict(box=box, halo=(wspan, 0, 0), groups=groups, taps=out_taps, n_tile=G * Np, a_bytes=a_bytes, resident=True,
                tail=tail, pitch=pitch, slabs=(G, 1, nslots))


def _make_conv_halo_plan(view, lay, a_channels, w_packed, Np, tile_space, out, out_f32, out_off, ostrides, bias,
                         accumulate, keep, stats=None, prologue=None) -> ConvHaloPlan:
    lib = L.load()
    d = L.ConvHaloDesc()
    keep = keep + _set_prologue(d, prologue, a_channels)
    d.amap = view
    d.a_channels = a_channels
    d.n_groups = len(lay["groups"])
    for i, g in enumerate(lay["groups"]):
        d.groups[i] = L.HaloGroup(*g)
    d.n_taps = len(lay["taps"])
    for i, (shift, k_off) in enumerate(lay["taps"]):
        d.taps[i] = L.HaloTap(shift, k_off)
    d.w_packed = w_packed.data_ptr()
    d.Np, d.Ktot, d.n_tile = Np, w_packed.shape[1], lay["n_tile"]
    d.Wt, d.Ht, d.Tt, d.Nt = tile_space
    d.bw, d.bh, d.bt, d.bn = lay["box"]
    d.halo_w, d.halo_h, d.halo_t = lay["halo"]
    d.out_bf16 = 0 if out is None else out.data_ptr()
    d.out_f32 = 0 if out_f32 is None else out_f32.data_ptr()
    d.out_off = out_off
    d.osw, d.osh, d.ost, d.osn = ostrides
    d.bias = 0 if bias is None else bias.data_ptr()
    d.accumulate = int(accumulate)
    d.allow_resident = int(lay["resident"])
    d.use_tail_boxes = int(bool(lay.get("tail", 0)))
    d.atom_pitch_rows = lay.get("pitch", 8)
    if lay.get("slabs"):
        d.slabs.n_slabs, d.slabs.axis, d.slabs.nslots = lay["slabs"]
    d.stats_partials = 0 if stats is None else stats.partials.data_ptr()
    d.stats_groups = 0 if stats is None else stats.groups
    h = C.c_void_p()
    L.check(lib.cstp_conv_halo_plan_create(C.byref(d), C.byref(h)))
    plan = ConvHaloPlan(h, lib.cstp_conv_halo_plan_destroy, keep + ((stats.partials,) if stats is not None else ()))
    plan.resident = bool(lib.cstp_conv_halo_plan_resident(h))
    if stats is not None:
        plan.stat_blocks = lib.cstp_conv_halo_plan_stat_blocks(h)
        if plan.stat_blocks * stats.groups * 2 * stats.Cp > stats.partials.numel():
            raise L.CstpError("BatchNorm partials buffer too small for the fused statistics")
    return plan


HALO_MIN_POSITIONS = 28 * 28      # per (t, n) slab: smaller extents cannot fill 128-row single-slab tiles


def conv_fwd_plan(x, w_packed, out, geom: ConvGeom, *, out_f32=None, bias=None, accumulate=False, n_tile=None,
                  box=None, allow_halo: bool = True, stats: "BNState | None" = None,
                  prologue: "BNState | None" = None) -> ConvPlan:
    """out[n,to,ho,wo,:] = conv3d(x, w) with x (N,T,H,W,Cp_in) bf16, w_packed [Np][taps*pad64(Cp_in)] bf16.
    With `stats` the kernel may also emit the BatchNorm statistics partials of `out` (plan.stat_blocks > 0 tells the caller
    to skip the separate statistics pass).  With `prologue` x is the RAW output of the producing convolution and the kernel
    convolves bf16(relu(x * prologue.scale + prologue.shift)) (include/cstp_b200.h cstp_prologue; the coefficients are
    read at run time, i.e. after the producer's cstp_bn_finalize of the same step)."""
    _require_cuda(x, w_packed, out, out_f32, bias)
    N, T, H, W, Ca = x.shape
    To, Ho, Wo = geom.out_dims(T, H, W)
    ref = out if out is not None else out_f32
    Np = ref.shape[-1]
    assert tuple(ref.shape[:4]) == (N, To, Ho, Wo), (ref.shape, (N, To, Ho, Wo))
    assert w_packed.shape[0] >= Np and w_packed.shape[1] == geom.taps * pad64(Ca), (w_packed.shape, Np, geom.taps, Ca)
    views, taps = _fwd_taps(x, geom)
    Kc = pad64(Ca)
    taps = [(m, dw, dh, dt, ti * Kc) for (m, dw, dh, dt, ti) in taps]
    ostr = (Np, Wo * Np, Ho * Wo * Np, To * Ho * Wo * Np)
    if allow_halo and box is None and n_tile is None and len(views) == 1 and Ho * Wo >= HALO_MIN_POSITIONS:
        lay = conv_halo_layout((Wo, Ho, To, N), [t[1:] for t in taps], Ca, Np)
        if lay is not None:
            # BatchNorm statistics fused into the epilogue: only for single 64-column N tiles, where every epilogue thread
            # can keep the running sum / sum of squares of its row's 64 columns in registers (no shuffles per tile).  The
            # first attempt (shuffle butterfly per 16-column chunk, all tile widths) removed 2.3 ms of bn_reduce passes at
            # batch 60 but cost 3-5 ms in the conv kernels and was taken out (profiles/README.md).
            fuse = (stats is not None and stats.groups in (1, 2) and N % stats.groups == 0
                    and out is not None and out_f32 is None and bias is None and not accumulate
                    and Np == 64 and lay["n_tile"] == 64 and lay["box"][3] == 1)
            return _make_conv_halo_plan(views[0], lay, Ca, w_packed, Np, (Wo, Ho, To, N), out, out_f32, 0, ostr, bias,
                                        accumulate, (x, w_packed, out, out_f32, bias), stats=stats if fuse else None,
                                        prologue=prologue)
    box = box or pick_box(Wo, Ho, To, N, 128)
    return _make_conv_plan(views, taps, Ca, w_packed, Np, (Wo, Ho, To, N), box, out, out_f32, 0, ostr, bias, accumulate,
                           n_tile, (x, w_packed, out, out_f32, bias), prologue=prologue)


def conv_dgrad_plans(g, wt_packed, dx, geom: ConvGeom, *, accumulate=False, allow_halo: bool = True) -> tuple[list[ConvPlan], bool]:
    """dx (N,T,H,W,Cp_in) = conv_transpose(g (N,To,Ho,Wo,Cp_out)); wt_packed [Cp_in][taps*pad64(Cp_out)] bf16.

    One plan per stride-parity class of dx.  Returns (plans, covers_all): when covers_all is False some classes
    receive no tap (1x1x1 strided conv) and dx must be zero-filled by the caller unless accumulating."""
    _require_cuda(g, wt_packed, dx)
    N, T, H, W, Ci = dx.shape
    _, To, Ho, Wo, Co = g.shape
    (kt, kh, kw), (st, sh, sw), (pt, ph, pw) = geom.kernel, geom.stride, geom.pad
    Kc = pad64(Co)
    assert wt_packed.shape[0] >= Ci and wt_packed.shape[1] == geom.taps * Kc
    gview = _view5(g)
    plans = []
    classes = dgrad_classes(tuple(dx.shape), geom)
    live = [cl for cl in classes if cl["taps"]]
    rest = []
    for cl in live:
        taps = [(0, dw_, dh_, dt_, ti * Kc) for (dw_, dh_, dt_, ti) in cl["taps"]]
        # the halo kernel takes the dgrad of stride-1 convolutions only: the stride-parity classes of a strided one run on
        # conv_gemm (measured at batch 60: conv3.block1.conv1.spatial dgrad 0.89 ms as one conv_gemm launch, 0.99 ms with
        # its 2- and 4-tap classes on the halo kernel)
        if allow_halo and tuple(geom.stride) == (1, 1, 1) and cl["space"][0] * cl["space"][1] >= HALO_MIN_POSITIONS:
            lay = conv_slab_layout(cl["space"], [t[1:] for t in taps], Co, Ci)
            if lay is None:
                lay = conv_halo_layout(cl["space"], [t[1:] for t in taps], Co, Ci)
            if lay is not None:
                plans.append(_make_conv_halo_plan(gview, lay, Co, wt_packed, Ci, cl["space"], dx, None, cl["off"],
                                                  cl["ostrides"], None, accumulate, (g, wt_packed, dx)))
                continue
        rest.append((cl, taps))
    if (1 < len(rest) <= 8
            and all(cl["space"] == rest[0][0]["space"] and cl["ostrides"] == rest[0][0]["ostrides"] for cl, _ in rest)
            and sum(len(t) for _, t in rest) <= L.CSTP_MAX_TAPS):
        # stride-parity classes that share their tile space (even extents): ONE launch, class-minor tile order -- the
        # classes of one tile read the same boxes of g at the same time
        taps, cls, t0 = [], [], 0
        for cl, tp in rest:
            taps += tp
            cls.append((t0, len(tp), cl["off"]))
            t0 += len(tp)
        cl0 = rest[0][0]
        plans.append(_make_conv_plan([gview], taps, Co, wt_packed, Ci, cl0["space"], pick_box(*cl0["space"], 128), dx, None,
                                     cl0["off"], cl0["ostrides"], None, accumulate, None, (g, wt_packed, dx), classes=cls))
    else:
        for cl, taps in rest:
            plans.append(_make_conv_plan([gview], taps, Co, wt_packed, Ci, cl["space"], pick_box(*cl["space"], 128), dx, None,
                                         cl["off"], cl["ostrides"], None, accumulate, None, (g, wt_packed, dx)))
    return plans, len(live) == len(classes)


def linear_plan(x, w_packed, out, *, out_f32=None, bias=None, accumulate=False) -> ConvPlan:
    """out[B][Np] = x[B][Cp] @ w^T (+bias): a 1-tap implicit GEMM over a (B,1,1,1,Cp) tensor."""
    B, Ca = x.shape
    ref = out if out is not None else out_f32
    Np = ref.shape[-1]
    x5 = x.view(1, 1, 1, B, Ca)
    o5 = None if out is None else out.view(1, 1, 1, B, Np)
    of5 = None if out_f32 is None else out_f32.view(1, 1, 1, B, Np)
    return conv_fwd_plan(x5, w_packed, o5, ConvGeom((1, 1, 1)), out_f32=of5, bias=bias, accumulate=accumulate,
                         box=(128, 1, 1, 1))


@dataclass
class WgradSpec:
    plan: WgradPlan
    n_mchunks: int
    Np: int
    chunk_tap: torch.Tensor
    chunk_coff: torch.Tensor
    cout: int
    cin: int
    taps: int
    partials: torch.Tensor
    layout: int = 0              # 1: the stem over cstp_stem_pack rows, dW is the reference's (cout, 3, 1, 7, 7) tensor;
    #                              2: transposed product (rows (tap, cout), columns cin)
    chunk_splits: torch.Tensor | None = None      # per-chunk number of split-K partials (M classes), None: plan.splits

    def run(self, dw: torch.Tensor, accumulate: bool = False):
        self.plan.run()
        L.check(L.load().cstp_wgrad_finalize(_ptr(self.partials), self.plan.splits, self.n_mchunks, self.Np,
                                             _ptr(self.chunk_tap), _ptr(self.chunk_coff), self.cout, self.cin,
                                             self.taps, _ptr(dw), int(accumulate), self.layout, _ptr(self.chunk_splits),
                                             _stream()))


class WgradHaloPlan(_Plan):
    splits: int = 1

    def run(self):
        L.check(L.load().cstp_wgrad_halo_plan_run(self.handle, _stream()))


def _wgrad_halo_side(m_channels: int, n_channels: int, dims, geom: ConvGeom, flip: bool, sms: int, xform: bool = False):
    """One orientation of the all-taps-per-CTA weight-gradient kernel: the operand with `m_channels` carries the taps (staged
    with a halo, M = (tap, 64-channel chunk)), the other one (`n_channels`, N axis) is staged as plain boxes.  flip: the M
    side is dL/d(raw) and the N side the activations (the taps then shift the other way).  Returns the layout dict with a
    `cost` (model cycles per K-block: the larger of tensor time and shared-memory time) or None."""
    (kt, kh, kw), (pt, ph, pw) = geom.kernel, geom.pad
    N, To, Ho, Wo = dims
    n_cc = pad64(m_channels) // 64
    n_chunks = geom.taps * n_cc
    if n_chunks > 32:
        return None
    n_mtiles = (n_chunks + 1) // 2
    Np = n_channels
    # full-width N tiles (every MMA as wide as the layer allows); the M tiles are dealt to CTA classes that fit TMEM
    n_ntiles = math.ceil(Np / 256)
    n_tile = pad16(math.ceil(Np / n_ntiles))
    if flip and xform and n_ntiles > 1:      # the prologue on the N-side boxes wants N-tile origins on 64-channel chunks
        n_tile = pad64(n_tile)
        n_ntiles = math.ceil(Np / n_tile)
    mt_per_class = min(n_mtiles, 512 // n_tile)
    n_mclasses = math.ceil(n_mtiles / mt_per_class)
    mt_per_class = math.ceil(n_mtiles / n_mclasses)          # balanced classes (5 tiles, cap 3 -> 3 + 2)
    if n_mclasses > 8:
        return None
    temporal = kt > 1
    # tap a reads the M-side operand at offset (a - pad) from the K-block origin -- or, flipped, at -(a - pad)
    off = (lambda a, k, p_: (k - 1 - a) if flip else a)
    org = (lambda k, p_: -(k - 1 - p_) if flip else -p_)
    # 1 x k x k filters, 2-D halo: ONE staged (8 + kw - 1) x (8 + kh - 1) box per 64-channel chunk serves every tap (a tap
    # is a whole-row shift of it; the 8 positions of a w run are one swizzle atom, atoms one box row apart).  The box is
    # then cheap enough to be re-staged by several CTA classes.
    halo_2d = (not temporal and kw > 1 and kh > 1 and n_ntiles * n_mclasses <= 6
               and math.ceil(Wo / 8) * math.ceil(Ho / 8) * 64 <= 1.35 * Wo * Ho)
    if n_ntiles * n_mclasses > 2 and not halo_2d:          # the M-side boxes are re-staged once per class
        return None
    pitch = 8
    if halo_2d:
        box, halo, pitch = (8, 8, 1, 1), (kw - 1, kh - 1, 0), 8 + kw - 1
        bw, bh, bt, _ = box
        xrows = (bw + halo[0]) * (bh + halo[1])
        xbox_bytes = (xrows * 128 + 1023) // 1024 * 1024
        xboxes = [(cc * 64, org(kw, pw), org(kh, ph), 0) for cc in range(n_cc)]
        chunks = [(cc * xbox_bytes + (off(b_, kh, ph) * pitch + off(c, kw, pw)) * 128, b_ * kw + c, cc * 64)
                  for b_ in range(kh) for c in range(kw) for cc in range(n_cc)]
    else:
        best = None
        for bw in (8, 16, 32, 64):
            for bh in (1, 2, 4, 8):
                for bt in ((1, 2, 4, 8) if temporal else (1,)):
                    if bw * bh * bt != 64:
                        continue
                    halo = (0, 0, kt - 1) if temporal else (0, kh - 1, 0)
                    tiles = math.ceil(Wo / bw) * math.ceil(Ho / bh) * math.ceil(To / bt)
                    staged = tiles * (bw + halo[0]) * (bh + halo[1]) * (bt + halo[2]) * (1 if temporal else kw)
                    key = (staged, -bw)
                    if best is None or key < best[0]:
                        best = (key, (bw, bh, bt, 1), halo)
        _, box, halo = best
        bw, bh, bt, _ = box
        xrows = (bw + halo[0]) * (bh + halo[1]) * (bt + halo[2])
        xbox_bytes = xrows * 128
        xboxes, chunks = [], []
        if temporal:
            for cc in range(n_cc):
                xboxes.append((cc * 64, 0, 0, org(kt, pt)))
            for a in range(kt):
                for cc in range(n_cc):
                    chunks.append((cc * xbox_bytes + off(a, kt, pt) * (bw * bh) * 128, a, cc * 64))
        else:
            for c in range(kw):
                for cc in range(n_cc):
                    xboxes.append((cc * 64, (pw - c) if flip else (c - pw), org(kh, ph), 0))
            for b_ in range(kh):
                for c in range(kw):
                    for cc in range(n_cc):
                        chunks.append(((c * n_cc + cc) * xbox_bytes + off(b_, kh, ph) * bw * 128, b_ * kw + c, cc * 64))
    if len(xboxes) > 16:
        return None
    chunks.sort()
    n_gboxes = math.ceil(n_tile / 64)
    stage = len(xboxes) * xbox_bytes + n_gboxes * 8192
    if 2 * stage + 1280 > SMEM_LIMIT:
        return None
    splits = max(1, sms // n_ntiles)
    kblocks = math.ceil(Wo / bw) * math.ceil(Ho / bh) * math.ceil(To / bt) * N
    splits = min(splits, kblocks)
    mmas = 4 * n_mtiles * n_ntiles
    cost = max(mmas * n_tile / 2, mmas * (4096 + 32 * n_tile) / 128)
    return dict(box=box, halo=halo, xboxes=xboxes, chunks=chunks, xbox_bytes=xbox_bytes, n_tile=n_tile,
                n_ntiles=n_ntiles, splits=splits, need=splits * n_chunks * 64 * Np, pitch=pitch,
                mt_per_class=mt_per_class if n_mclasses > 1 else 0, flip=flip, cost=cost)


def wgrad_halo_layout(x_shape, g_shape, geom: ConvGeom, sms: int = 148, xform: bool = False):
    """Geometry of the all-taps-per-CTA weight-gradient kernel (csrc/wgrad_halo.cu) for a stride-1 1xkxk / kx1x1
    convolution, or None when the layer does not qualify (then csrc/wgrad.cu is used).  Pure shape arithmetic.

    Two orientations are costed (shared-memory bytes and tensor cycles per K-block) and the cheaper one is taken: the taps
    ride on X (M = (tap, cin chunk), N = cout) or -- `flip`, same-size convolutions only -- on dL/d(raw)
    (M = (tap, cout chunk), N = cin), which keeps the MMAs wide for the 144 -> 64 3x1x1 layers.

    Returns dict(box, halo, xboxes [(c_off, dw, dh, dt)] of the M-side tensor, chunks [(stage byte offset, tap index,
    first M-side channel)] sorted by offset, xbox_bytes, n_tile, n_ntiles, mt_per_class, splits, need (floats of split-K
    partials), flip).  xform: X is read through the operand prologue (constrains the N tiles of the flipped form)."""
    (kt, kh, kw) = geom.kernel
    if tuple(geom.stride) != (1, 1, 1) or geom.taps == 1 or (kt > 1 and (kh > 1 or kw > 1)):
        return None
    N, T, H, W, Ca = x_shape
    _, To, Ho, Wo, Np = g_shape
    lay = _wgrad_halo_side(Ca, Np, (N, To, Ho, Wo), geom, False, sms, xform)
    if (T, H, W) == (To, Ho, Wo) and geom.pad_hi is None:
        alt = _wgrad_halo_side(Np, Ca, (N, To, Ho, Wo), geom, True, sms, xform)
        if alt is not None and (lay is None or alt["cost"] < lay["cost"]):
            lay = alt
    return lay


def wgrad_partials_need(x_shape, g_shape, geom: ConvGeom, sms: int = 148) -> int:
    """Upper bound (floats) of the split-K scratch wgrad_plan needs for this layer."""
    lays = [wgrad_halo_layout(x_shape, g_shape, geom, sms, xf) for xf in (False, True)]
    if lays[0] is not None:
        return max(l["need"] for l in lays if l is not None)
    Ca, Np = x_shape[-1], g_shape[-1]
    nch = geom.taps * (pad64(Ca) // 64)
    To, Ho, Wo = g_shape[1:4]
    box = pick_box(Wo, Ho, To, g_shape[0], 64)
    kblocks = math.ceil(Wo / box[0]) * math.ceil(Ho / box[1]) * math.ceil(To / box[2]) * math.ceil(g_shape[0] / box[3])
    return max(_wgrad_gemm_shape(nch, Np, kblocks, sms, xf)[2] for xf in (False, True)) * nch * 64 * Np


def _wgrad_gemm_shape(nch: int, Np: int, kblocks: int, sms: int = 148, xform: bool = False) -> tuple[int, int, int]:
    """(n_tile, mt_per_cta, splits) of csrc/wgrad.cu for `nch` 64-row M chunks, Np columns and `kblocks` 64-position K-blocks.
    The kernel is bound by the L2 -> SM feed: a CTA stages 2 * mt X boxes and n_tile / 64 G boxes of 8 KB per K-block, so
      * the N tile is the multiple of 64 that needs the fewest tiles, then the fewest padded columns (576 -> 3 x 192, not
        256 + 256 + 64 with every MMA 256 wide);
      * a CTA takes as many 128-row M tiles as TMEM (mt * n_tile <= 512 columns) and a three-stage pipeline allow: they
        share one staged G tile (the prologue variant takes one: its transform keeps the coefficients of two boxes in
        registers);
      * the split-K factor minimises waves x K-blocks per split + the cost of writing and re-reading one more partial."""
    if Np <= 256:
        n_tile = Np
    else:
        n_tile = min((256, 192, 128), key=lambda c: (math.ceil(Np / c), math.ceil(Np / c) * c, -c))
    ngb = math.ceil(n_tile / 64)
    mt = 1
    for m in range(2, 5):                                        # csrc/wgrad.cu takes up to four M tiles per CTA
        if m * n_tile <= 512 and 3 * (2 * m + ngb) * 8192 <= SMEM_BUDGET and m <= math.ceil(nch / 2):
            mt = m
    # (the split-K factor is the plain kernel's also behind the prologue, which runs one M tile per CTA: the same K ranges
    # summed in the same order keep the fused edge bit-identical to bn_apply followed by the plain kernel)
    base = math.ceil(nch / (2 * mt)) * math.ceil(Np / n_tile)
    t_kb = (2 * mt + ngb) * 195.0 / 1.7e9                        # seconds per K-block and CTA at the L2 fair share
    t_part = 2.0 * nch * 64 * Np * 4 / 5e12                      # one more partial: written here, read by the finalize pass
    best = None
    for sp in range(1, max(1, min(kblocks // 4, math.ceil(4 * sms / base))) + 1):
        cost = math.ceil(base * sp / sms) * math.ceil(kblocks / sp) * t_kb + sp * t_part
        if best is None or cost < best[0] - 1e-12:
            best = (cost, sp)
    return n_tile, 1 if xform else mt, best[1]


def wgrad_plan(x, g, geom: ConvGeom, cout: int, cin: int, partials: torch.Tensor, *, splits: int | None = None,
               box=None, sms: int = 148, allow_halo: bool = True, prologue: "BNState | None" = None,
               layout: int = 0) -> WgradSpec:
    """dW (cout, cin, kt, kh, kw) from x (N,T,H,W,Cp_in) and g (N,To,Ho,Wo,Cp_out); `partials` is fp32 scratch.
    With `prologue` x is the raw output of the producing convolution (see conv_fwd_plan).  layout = 1: x holds the stem's
    packed row pairs (stem_pack), geom is STEM_GEOM, cin = 64 and dW the reference's (cout, 3, 1, 7, 7) weight gradient."""
    _require_cuda(x, g, partials)
    lib = L.load()
    N, T, H, W, Ca = x.shape
    _, To, Ho, Wo, Np = g.shape
    assert geom.out_dims(T, H, W) == (To, Ho, Wo)
    dev = x.device
    lay = (wgrad_halo_layout(tuple(x.shape), tuple(g.shape), geom, sms, prologue is not None)
           if (allow_halo and splits is None and box is None) else None)
    if lay is not None:
        flip = lay["flip"]
        if layout != 0 and flip:
            raise L.CstpError("the stem weight-gradient layout has no transposed form")
        d = L.WgradHaloDesc()
        d.xmap, d.gmap = (_view5(g), _view5(x)) if flip else (_view5(x), _view5(g))
        if flip:
            Np = Ca                       # the N axis (columns of the partials) is cin
        d.mt_per_class = lay["mt_per_class"]
        d.pro_on_b = int(flip)
        d.n_xboxes = len(lay["xboxes"])
        for i, xb in enumerate(lay["xboxes"]):
            d.xboxes[i] = L.XBox(*xb)
        d.n_chunks = len(lay["chunks"])
        for i, (off, _, _) in enumerate(lay["chunks"]):
            d.chunk_off[i] = off
        d.Np, d.n_tile = Np, lay["n_tile"]
        d.Wt, d.Ht, d.Tt, d.Nt = Wo, Ho, To, N
        d.bw, d.bh, d.bt, d.bn = lay["box"]
        d.halo_w, d.halo_h, d.halo_t = lay["halo"]
        d.splits = lay["splits"]
        d.atom_pitch_rows = lay.get("pitch", 8)
        if partials.numel() < lay["need"]:
            raise L.CstpError(f"wgrad partials scratch too small: {partials.numel()} < {lay['need']}")
        d.partials = partials.data_ptr()
        keep = _set_prologue(d, prologue, Ca)
        h = C.c_void_p()
        L.check(lib.cstp_wgrad_halo_plan_create(C.byref(d), C.byref(h)))
        plan = WgradHaloPlan(h, lib.cstp_wgrad_halo_plan_destroy, (x, g, partials) + keep)
        plan.splits = lib.cstp_wgrad_halo_plan_splits(h)
        chunk_splits = None
        if lay["mt_per_class"]:
            cs = (C.c_int32 * len(lay["chunks"]))()
            L.check(lib.cstp_wgrad_halo_plan_chunk_splits(h, cs, len(lay["chunks"])))
            chunk_splits = torch.tensor(list(cs), dtype=torch.int32, device=dev)
        return WgradSpec(plan, len(lay["chunks"]), Np,
                         torch.tensor([c[1] for c in lay["chunks"]], dtype=torch.int32, device=dev),
                         torch.tensor([c[2] for c in lay["chunks"]], dtype=torch.int32, device=dev), cout, cin, geom.taps,
                         partials, 2 if flip else layout, chunk_splits)
    views, taps = _fwd_taps(x, geom)
    nchunk_c = pad64(Ca) // 64
    mch, ctap, ccoff = [], [], []
    for (m, dw_, dh_, dt_, ti) in taps:
        for cc in range(nchunk_c):
            mch.append((m, dw_, dh_, dt_, cc * 64))
            ctap.append(ti)
            ccoff.append(cc * 64)
    if len(mch) > L.CSTP_MAX_MCHUNKS:
        raise L.CstpError(f"wgrad needs {len(mch)} M chunks > {L.CSTP_MAX_MCHUNKS}")
    box = box or pick_box(Wo, Ho, To, N, 64)
    kblocks = math.ceil(Wo / box[0]) * math.ceil(Ho / box[1]) * math.ceil(To / box[2]) * math.ceil(N / box[3])
    n_tile, n_mt, auto_splits = _wgrad_gemm_shape(len(mch), Np, kblocks, sms, prologue is not None)
    if splits is None:
        splits = auto_splits
    d = L.WgradDesc()
    d.n_amaps = len(views)
    for i, v in enumerate(views):
        d.amap[i] = v
    d.n_mchunks = len(mch)
    for i, mc in enumerate(mch):
        d.mchunks[i] = L.MChunk(*mc)
    d.gmap = _view5(g)
    d.Np, d.n_tile, d.mt_per_cta = Np, n_tile, n_mt
    d.Wt, d.Ht, d.Tt, d.Nt = Wo, Ho, To, N
    d.bw, d.bh, d.bt, d.bn = box
    d.splits = splits
    need = splits * len(mch) * 64 * Np
    if partials.numel() < need:
        raise L.CstpError(f"wgrad partials scratch too small: {partials.numel()} < {need}")
    d.partials = partials.data_ptr()
    keep = _set_prologue(d, prologue, Ca)
    h = C.c_void_p()
    L.check(lib.cstp_wgrad_plan_create(C.byref(d), C.byref(h)))
    plan = WgradPlan(h, lib.cstp_wgrad_plan_destroy, (x, g, partials) + keep)
    plan.splits = lib.cstp_wgrad_plan_splits(h)
    return WgradSpec(plan, len(mch), Np, torch.tensor(ctap, dtype=torch.int32, device=dev),
                     torch.tensor(ccoff, dtype=torch.int32, device=dev), cout, cin, geom.taps, partials, layout)


# ------------------------------------------------------------------------------------------------ thin wrappers
def _pack_dims(w: torch.Tensor, transpose) -> tuple[int, int, int]:
    """(cout, cin, taps) as the pack kernels index them; transpose = 2 is the stem over packed row pairs: 64 pixel channels
    (hpar, kw, c), 4 row-pair taps of a (cout, 3, 1, 7, 7) weight."""
    if int(transpose) == 2:
        if tuple(w.shape[1:]) != (3, 1, 7, 7):
            raise L.CstpError(f"stem weight layout expects (cout, 3, 1, 7, 7), got {tuple(w.shape)}")
        return w.shape[0], STEM_CHANNELS, 4
    cout, cin = w.shape[0], w.shape[1]
    return cout, cin, w.numel() // (cout * cin)


def pack_weight(w: torch.Tensor, packed: torch.Tensor, *, transpose=False) -> None:
    """fp32 (cout, cin, *kernel) -> bf16 packed [Rp][taps*Kc] (forward), its dgrad transpose, or (transpose = 2) the stem
    layout packed[co][kh*Kc + kw*3 + c]."""
    _require_cuda(w, packed)
    cout, cin, taps = _pack_dims(w, transpose)
    Rp, Ktot = packed.shape
    L.check(L.load().cstp_pack_weight(_ptr(w), cout, cin, taps, int(transpose), _ptr(packed), Rp, Ktot // taps, _stream()))


class PackList:
    """A fixed list of (fp32 weight, bf16 packed, transpose) jobs executed as ONE launch (cstp_pack_weights_batched)."""

    def __init__(self, jobs, device):
        rows, prefix, total = [], [0], 0
        for w, packed, transpose in jobs:
            _require_cuda(w, packed)
            cout, cin, taps = _pack_dims(w, transpose)
            Rp, Ktot = packed.shape
            # (the kernel writes eight K columns per 16-byte store)
            if (Ktot // taps) % 8 or Ktot % taps or packed.data_ptr() % 16 or not packed.is_contiguous():
                raise L.CstpError(f"packed weight {tuple(packed.shape)} / {taps} taps: K rows must be 16-byte aligned multiples of 8")
            rows.append([w.data_ptr(), packed.data_ptr(), cout, cin, taps, int(transpose), Rp, Ktot // taps])
            total += Rp * Ktot
            prefix.append(total)
        self.n, self.total = len(rows), total
        self.jobs = torch.tensor(rows, dtype=torch.int64, device=device)
        self.prefix = torch.tensor(prefix, dtype=torch.int64, device=device)
        self._keep = jobs

    def run(self) -> None:
        if self.n:
            L.check(L.load().cstp_pack_weights_batched(_ptr(self.jobs), _ptr(self.prefix), self.n, self.total, _stream()))


# The 1x7x7 s(1,2,2) p(0,3,3) stem (r21d_byol.py:198) over stem_pack row pairs: output row ho reads the four row pairs
# ho - 2 .. ho + 1 (frame rows 2*ho - 4 .. 2*ho + 3; the filter has no element for the first), stride 1.
STEM_GEOM = ConvGeom((1, 4, 1), (1, 1, 1), (0, 2, 0), (0, 1, 0))
STEM_CHANNELS = 64          # two frame rows x (21 packed (kw, c) channels zero-padded to 32)


def stem_pack(x: torch.Tensor, P: torch.Tensor) -> None:
    """fp32 NCDHW clips (N,3,T,H,W) -> bf16 P (N,T,H/2,W/2,64),
    P[n][t][h2][wo][hpar*32 + kw*3 + c] = x[n][c][t][2*h2 + hpar][2*wo + kw - 3]."""
    _require_cuda(x, P)
    N, Cc, T, H, W = x.shape
    assert Cc == 3 and x.dtype == torch.float32 and x.is_contiguous()
    assert tuple(P.shape) == (N, T, H // 2, W // 2, STEM_CHANNELS) and P.is_contiguous()
    L.check(L.load().cstp_stem_pack(_ptr(x), N, T, H, W, _ptr(P), _stream()))


BN_REDUCE_CTAS_PER_SM = 2         # per statistics group (co-residency sweep: profiles/r01_overlap_sweep.txt)


def bn_nblocks(rows_per_group: int, Cp: int, sms: int = 148) -> int:
    rows_per_pass = max(1, 256 // min(Cp // 8, 128))
    return max(1, min(BN_REDUCE_CTAS_PER_SM * sms, math.ceil(rows_per_group / (rows_per_pass * 8))))


@dataclass
class BNState:
    """Per-call BatchNorm scratch: statistics partials, affine coefficients and saved mean/invstd."""
    C: int
    Cp: int
    groups: int
    nblocks: int
    partials: torch.Tensor
    scale: torch.Tensor
    shift: torch.Tensor
    mean: torch.Tensor
    invstd: torch.Tensor
    coef: torch.Tensor = field(default=None)
    compact: torch.Tensor = field(default=None)      # [groups][2][Cp] row exchanged by world-synchronised BatchNorm

    @staticmethod
    def alloc(C_: int, Cp: int, groups: int, rows_per_group: int, device, backward: bool = True) -> "BNState":
        nb = bn_nblocks(rows_per_group, Cp)
        f = dict(dtype=torch.float32, device=device)
        # (room for the fused-statistics path too: one partial row per CTA of a persistent conv kernel, <= 148 + slack)
        return BNState(C_, Cp, groups, nb, torch.empty(max(nb, 160) * groups * 2 * Cp, **f), torch.empty(groups * Cp, **f),
                       torch.empty(groups * Cp, **f), torch.empty(groups * Cp, **f), torch.empty(groups * Cp, **f),
                       torch.empty(groups * 3 * Cp, **f) if backward else None, torch.empty(groups * 2 * Cp, **f))


def bn_forward_stats(raw, st: BNState, gamma, beta, running_mean, running_var, eps=1e-5, momentum=0.1,
                     fused_blocks: int = 0, sync=None) -> None:
    """Batch statistics of raw -> scale/shift/mean/invstd (+ running buffers).  fused_blocks > 0: the producing conv
    kernel already wrote that many partial rows into st.partials (no statistics pass over raw).  `sync` (an object with
    `.world` and `.all_reduce(tensor)`) makes the statistics span every rank (SyncBN over the data-parallel group): the
    per-rank sums are collapsed to one row, summed across ranks and finalized with the global row count."""
    rows = raw.numel() // st.Cp
    lib = L.load()
    nblocks = fused_blocks or st.nblocks
    if not fused_blocks:
        L.check(lib.cstp_bn_stats(_ptr(raw), rows, st.Cp, st.groups, _ptr(st.partials), st.nblocks, _stream()))
    partials, rpg = st.partials, rows // st.groups
    if sync is not None and sync.world > 1:
        L.check(lib.cstp_bn_partials_reduce(_ptr(st.partials), nblocks, st.groups, st.Cp, _ptr(st.compact), _stream()))
        sync.all_reduce(st.compact)
        partials, nblocks, rpg = st.compact, 1, rpg * sync.world
    L.check(lib.cstp_bn_finalize(_ptr(partials), nblocks, st.groups, rpg, st.C, st.Cp, _ptr(gamma),
                                 _ptr(beta), eps, momentum, _ptr(running_mean), _ptr(running_var), _ptr(st.scale),
                                 _ptr(st.shift), _ptr(st.mean), _ptr(st.invstd), _stream()))


def bn_apply(raw, st: BNState, out, *, relu: bool, res=None, res_state: BNState | None = None,
             res_relu: bool = False) -> None:
    """out = [relu](raw*scale + shift [+ shortcut]).  The shortcut is `res` itself, or -- with res_state -- the BatchNorm
    output res*scale2 + shift2 of a raw conv output (downsample branch), or -- with res_relu as well -- the BatchNorm + ReLU
    activation bf16(relu(res*scale2 + shift2)) that was never written out (fused-prologue edges)."""
    rows = raw.numel() // st.Cp
    mode = 0 if res is None else ((3 if res_relu else 2) if res_state is not None else 1)
    L.check(L.load().cstp_bn_apply(_ptr(raw), rows, st.Cp, st.groups, _ptr(st.scale), _ptr(st.shift), int(relu), mode,
                                   _ptr(res), _ptr(res_state.scale if res_state else None),
                                   _ptr(res_state.shift if res_state else None), _ptr(out), _stream()))


def bn_backward(d, act, raw, st: BNState, gamma, dgamma, dbeta, g_out, *, dz=None, accumulate=False,
                mask_from_raw: bool = False, sync=None) -> None:
    """g_out = dL/d(raw) given d = dL/d(act); fills dgamma/dbeta.  The ReLU mask is `act > 0` when act is given, or --
    with mask_from_raw -- recomputed as raw*scale + shift > 0 from the forward coefficients kept in `st` (the same fmaf
    the forward apply evaluated; saves reading act twice)."""
    rows = raw.numel() // st.Cp
    lib = L.load()
    ms, mb = (st.scale, st.shift) if mask_from_raw else (None, None)
    if mask_from_raw:
        act = None
    L.check(lib.cstp_bn_bwd_reduce(_ptr(d), _ptr(act), _ptr(raw), rows, st.Cp, st.groups, _ptr(st.mean),
                                   _ptr(st.invstd), _ptr(ms), _ptr(mb), _ptr(st.partials), st.nblocks, _stream()))
    if sync is not None and sync.world > 1:
        # SyncBN backward: dgamma / dbeta stay this rank's local sums (the data-parallel gradient mean combines them),
        # the dx coefficients use the sums over every rank and the global row count
        L.check(lib.cstp_bn_partials_reduce(_ptr(st.partials), st.nblocks, st.groups, st.Cp, _ptr(st.compact), _stream()))
        L.check(lib.cstp_bn_bwd_finalize(_ptr(st.compact), 1, st.groups, rows // st.groups, st.C, st.Cp, _ptr(gamma),
                                         _ptr(st.mean), _ptr(st.invstd), _ptr(dgamma), _ptr(dbeta), int(accumulate),
                                         _ptr(st.coef), _stream()))
        sync.all_reduce(st.compact)
        L.check(lib.cstp_bn_bwd_finalize(_ptr(st.compact), 1, st.groups, (rows // st.groups) * sync.world, st.C, st.Cp,
                                         _ptr(gamma), _ptr(st.mean), _ptr(st.invstd), None, None, 0, _ptr(st.coef),
                                         _stream()))
    else:
        L.check(lib.cstp_bn_bwd_finalize(_ptr(st.partials), st.nblocks, st.groups, rows // st.groups, st.C, st.Cp,
                                         _ptr(gamma), _ptr(st.mean), _ptr(st.invstd), _ptr(dgamma), _ptr(dbeta),
                                         int(accumulate), _ptr(st.coef), _stream()))
    L.check(lib.cstp_bn_bwd_apply(_ptr(d), _ptr(act), _ptr(raw), rows, st.Cp, st.groups, _ptr(st.mean), _ptr(st.invstd),
                                  _ptr(st.coef), _ptr(ms), _ptr(mb), _ptr(g_out), _ptr(dz), _stream()))


def avgpool_fwd(x, out_f32, out_bf16, rows_out: int | None = None, ld_out: int | None = None) -> None:
    N = x.shape[0]
    Cp = x.shape[-1]
    P = x.numel() // (N * Cp)
    L.check(L.load().cstp_avgpool_fwd(_ptr(x), N, P, Cp, _ptr(out_f32), _ptr(out_bf16), rows_out or N, ld_out or Cp,
                                      _stream()))


def avgpool_bwd(dfeat, dx, dcat=None) -> None:
    N = dx.shape[0]
    Cp = dx.shape[-1]
    P = dx.numel() // (N * Cp)
    rows_cat, ld_cat = (dcat.shape[0], dcat.shape[1]) if dcat is not None else (0, 0)
    L.check(L.load().cstp_avgpool_bwd(_ptr(dfeat), _ptr(dcat), rows_cat, ld_cat, N, P, Cp, _ptr(dx), _stream()))


def colsum(x, C_: int, out, accumulate=False) -> None:
    rows, Cp = x.shape
    L.check(L.load().cstp_colsum(_ptr(x), rows, Cp, C_, _ptr(out), int(accumulate), _stream()))


def cast_pad(x, out, cols: int | None = None, scale_dev=None) -> None:
    rows, ld_in = x.shape
    L.check(L.load().cstp_cast_pad(_ptr(x), rows, cols or ld_in, ld_in, _ptr(out), out.shape[1], _ptr(scale_dev),
                                   _stream()))


def byol_loss(pred, tproj, B: int, D: int, loss_out, upstream=None, dpred=None) -> None:
    L.check(L.load().cstp_byol_loss(_ptr(pred), _ptr(tproj), B, D, pred.shape[1], _ptr(loss_out), _ptr(upstream),
                                    _ptr(dpred), _stream()))


REPR_DIM, REPR_MAX_ROWS = 512, 8192
REPR_STATS = ("std_feat", "std_proj", "std_pred", "std_tproj", "feat_norm")     # the columns of one view's statistics


def _check_repr_stats(blocks, B: int, out) -> None:
    if not 2 <= B <= REPR_MAX_ROWS:
        raise L.CstpError(f"repr_stats: B = {B}, expected 2 .. {REPR_MAX_ROWS} (an unbiased std needs two rows per view)")
    for t in blocks:
        if t is None:
            continue
        if t.dtype != torch.float32 or t.dim() != 2 or t.stride(1) != 1 or t.shape[0] < 2 * B \
                or t.shape[1] < REPR_DIM or t.stride(0) < REPR_DIM:
            raise L.CstpError(f"repr_stats: row blocks must be fp32 [2B][ld >= {REPR_DIM}] with unit column stride, got "
                              f"{t.dtype} {tuple(t.shape)} strides {t.stride()} for B = {B}")
    if out.dtype != torch.float32 or not out.is_contiguous() or out.numel() < 2 * len(REPR_STATS):
        raise L.CstpError("repr_stats: out must be contiguous fp32 [2][5]")


def repr_stats(feat, proj, pred, tproj, B: int, out) -> None:
    """Representation (collapse) statistics of one step into out fp32 [2][5]: per view, the mean over 512 columns of the
    unbiased std over the view's B rows of the l2-normalised online pooled feature / projector / predictor / target
    projector output (REPR_STATS order), and the feature's mean row norm.  Each block is fp32 [2B][ld] (views stacked
    along the rows, the first 512 columns valid) or None (skipped: its entry is 0).  Exact arithmetic of
    include/cstp_b200.h cstp_repr_stats."""
    blocks = (feat, proj, pred, tproj)
    _check_repr_stats(blocks, B, out)
    _require_cuda(*blocks, out)
    ld = [0 if t is None else t.stride(0) for t in blocks]
    L.check(L.load().cstp_repr_stats(_ptr(feat), ld[0], _ptr(proj), ld[1], _ptr(pred), ld[2], _ptr(tproj), ld[3], B,
                                     _ptr(out), _stream()))


def pretext_ce(logits, labels, dlogits, B: int, n_cls: int, weights5, losses_out) -> None:
    arr = C.c_void_p * 6
    lg = arr(*[t.data_ptr() for t in logits])
    lb = arr(*[t.data_ptr() for t in labels])
    dl = arr(*[0 if t is None else t.data_ptr() for t in dlogits]) if dlogits is not None else None
    L.check(L.load().cstp_pretext_ce(lg, lb, dl, B, n_cls, logits[0].shape[1], _ptr(weights5), _ptr(losses_out),
                                     _stream()))


def ntxent_workspace_floats(rows: int, d: int) -> int:
    """Scratch size (fp32 elements) that lets cstp_ntxent use its tensor-core path."""
    return max(int(L.load().cstp_ntxent_workspace_floats(rows, d)), 3 * rows + rows * d)


def ntxent(z, temperature: float, use_cosine: bool, loss_out, dz, workspace) -> None:
    rows, d = z.shape
    L.check(L.load().cstp_ntxent(_ptr(z), rows, d, float(temperature), int(use_cosine), _ptr(loss_out), _ptr(dz),
                                 _ptr(workspace), workspace.numel(), _stream()))


def l2norm_fwd(x, y_bf16, norms, d: int, eps: float = 1e-12) -> None:
    L.check(L.load().cstp_l2norm_fwd(_ptr(x), x.shape[0], d, x.shape[1], float(eps), _ptr(y_bf16), y_bf16.shape[1],
                                     _ptr(norms), _stream()))


def l2norm_bwd(x, norms, g_bf16, dx, d: int) -> None:
    L.check(L.load().cstp_l2norm_bwd(_ptr(x), _ptr(norms), _ptr(g_bf16), x.shape[0], d, x.shape[1], g_bf16.shape[1],
                                     _ptr(dx), _stream()))


def ce_loss(logits, labels, n_cls: int, loss_out, dlogits, workspace) -> None:
    L.check(L.load().cstp_ce_loss(_ptr(logits), _ptr(labels), logits.shape[0], n_cls, logits.shape[1], _ptr(loss_out),
                                  _ptr(dlogits), _ptr(workspace), _stream()))


def bn_eval_coeffs(st: BNState, gamma, beta, running_mean, running_var, eps: float = 1e-5) -> None:
    L.check(L.load().cstp_bn_eval_coeffs(_ptr(gamma), _ptr(beta), _ptr(running_mean), _ptr(running_var), st.C, st.Cp,
                                         st.groups, float(eps), _ptr(st.scale), _ptr(st.shift), _stream()))


def video_accumulate(logits, n_cls: int, seg, sums, rows: int | None = None) -> None:
    """sums[slot] += logits[first:first + count, :n_cls] in row order for every {slot, first, count} row of the int32
    device table seg [n][3] (count <= 0: skipped).  rows: how many leading rows of logits entries may name."""
    _require_cuda(logits, seg, sums)
    L.check(L.load().cstp_video_accumulate(_ptr(logits), rows or logits.shape[0], logits.shape[1], n_cls, _ptr(seg),
                                           seg.shape[0], _ptr(sums), sums.shape[0], _stream()))


def video_finalize(sums, fin, topk_out, labels=None, mean_out=None, hits=None) -> None:
    """For every {slot, count, video} row of the int32 device table fin [n][3]: mean = sums[slot] / count ->
    mean_out[video] (optional), topk_out[video] (int64 [videos][k]: descending, ties to the lower class), hits[0] / hits[1]
    += top-1 / top-5 hits against labels[video] (int64, optional); the slot is zeroed."""
    _require_cuda(sums, fin, topk_out, labels, mean_out, hits)
    n_slots, n_cls = sums.shape
    L.check(L.load().cstp_video_finalize(_ptr(sums), n_slots, n_cls, _ptr(fin), fin.shape[0], topk_out.shape[0],
                                         topk_out.shape[1], _ptr(labels), _ptr(mean_out), _ptr(topk_out), _ptr(hits),
                                         _stream()))


KNN_MAX_K, KNN_MAX_SPLITS, KNN_QUERY_TILE, KNN_CTAS_PER_SM = 64, 32, 64, 3


def knn_splits(nq: int, ng: int, sms: int = 148) -> int:
    """Gallery splits of cstp_knn_partial for nq queries against ng gallery rows: the count (at most 32, at least 512
    gallery rows each) whose grid of query tiles x splits leaves the least of its last wave of 148 x 3 resident CTAs
    idle; ties go to fewer splits (less merge work).  Results do not depend on it."""
    tiles, slots = -(-nq // KNN_QUERY_TILE), sms * KNN_CTAS_PER_SM
    best, best_eff = 1, 0.0
    for s in range(1, max(1, min(KNN_MAX_SPLITS, ng // 512)) + 1):
        ctas = tiles * s
        eff = ctas / (-(-ctas // slots) * slots)
        if eff > best_eff + 1e-9:
            best, best_eff = s, eff
    return best


def l2_normalize_rows(x, y) -> None:
    """y[n][d] = x[:, :d] / max(||x[:, :d]||, 1e-12) (F.normalize) for x fp32 [n][ld], y fp32 [n][d] contiguous."""
    _require_cuda(x, y)
    if x.dtype != torch.float32 or y.dtype != torch.float32 or x.stride(1) != 1 or not y.is_contiguous() \
            or x.shape[0] != y.shape[0] or x.shape[1] < y.shape[1]:
        raise L.CstpError("l2_normalize_rows: x fp32 [n][>= d] with unit column stride, y contiguous fp32 [n][d]")
    L.check(L.load().cstp_l2_normalize_rows(_ptr(x), x.shape[0], y.shape[1], x.stride(0), _ptr(y), _stream()))


def knn_partial(q, g, k: int, splits: int, part_val, part_idx) -> None:
    """Each gallery split's top-k of s(q, g) for normalised rows q [nq][d], g [ng][d] into part_val fp32 /
    part_idx int32 [splits][nq][k] (similarity descending, then the lower gallery index; -inf / -1 past the split)."""
    _require_cuda(q, g, part_val, part_idx)
    if q.dtype != torch.float32 or g.dtype != torch.float32 or not (q.is_contiguous() and g.is_contiguous()) \
            or q.shape[1] != g.shape[1] or part_val.dtype != torch.float32 or part_idx.dtype != torch.int32 \
            or part_val.shape != (splits, q.shape[0], k) or part_idx.shape != part_val.shape:
        raise L.CstpError("knn_partial: contiguous fp32 q [nq][d], g [ng][d]; part_val fp32 / part_idx int32 "
                          "[splits][nq][k]")
    L.check(L.load().cstp_knn_partial(_ptr(q), q.shape[0], _ptr(g), g.shape[0], q.shape[1], k, splits, _ptr(part_val),
                                      _ptr(part_idx), _stream()))


def knn_merge(part_val, part_idx, idx_out, sim_out, q_labels=None, g_labels=None, cutoffs=None, hits=None) -> None:
    """Merges knn_partial's lists into idx_out int64 / sim_out fp32 [nq][k]; with hits (int64 [len(cutoffs)]):
    hits[c] += queries with a label match among their first cutoffs[c] neighbours.  g_labels (int64) must hold one label
    per gallery row knn_partial searched."""
    _require_cuda(part_val, part_idx, idx_out, sim_out, q_labels, g_labels, cutoffs, hits)
    splits, nq, k = part_val.shape
    if part_idx.shape != part_val.shape or idx_out.dtype != torch.int64 or sim_out.dtype != torch.float32 \
            or idx_out.shape != (nq, k) or sim_out.shape != (nq, k) or not (idx_out.is_contiguous() and sim_out.is_contiguous()):
        raise L.CstpError("knn_merge: idx_out int64 / sim_out fp32 contiguous [nq][k] for the partial lists' nq, k")
    if hits is not None and (q_labels is None or g_labels is None or cutoffs is None or q_labels.dtype != torch.int64
                             or q_labels.numel() != nq or g_labels.dtype != torch.int64 or cutoffs.dtype != torch.int32
                             or hits.dtype != torch.int64 or hits.numel() != cutoffs.numel()):
        raise L.CstpError("knn_merge: int64 q_labels [nq] and g_labels, int32 cutoffs, int64 hits [len(cutoffs)]")
    L.check(L.load().cstp_knn_merge(_ptr(part_val), _ptr(part_idx), nq, k, splits, _ptr(idx_out), _ptr(sim_out),
                                    _ptr(q_labels), _ptr(g_labels), _ptr(cutoffs), 0 if cutoffs is None else cutoffs.numel(),
                                    _ptr(hits), _stream()))


def ema_update(k, q, m: float) -> None:
    import numpy as np
    L.check(L.load().cstp_ema_update(_ptr(k), _ptr(q), k.numel(), float(np.float32(m)), float(np.float32(1.0 - m)),
                                     _stream()))


def sgd_clip_step(p, g, mom, lr, momentum, wd, max_norm, do_clip, first_step, norm_out, workspace) -> None:
    L.check(L.load().cstp_sgd_clip_step(_ptr(p), _ptr(g), _ptr(mom), p.numel(), float(lr), float(momentum), float(wd),
                                        float(max_norm), int(do_clip), int(first_step), _ptr(norm_out), _ptr(workspace),
                                        _stream()))


def sgd_clip_step_dev(p, g, mom, hyper, norm_out, workspace) -> None:
    """sgd_clip_step with {lr, momentum, wd, max_norm, do_clip, first_step} read from the device vector `hyper` at run time
    (the form a captured CUDA graph replays while the host follows the learning-rate schedule)."""
    L.check(L.load().cstp_sgd_clip_step_dev(_ptr(p), _ptr(g), _ptr(mom), p.numel(), _ptr(hyper), _ptr(norm_out),
                                            _ptr(workspace), _stream()))


ADAM_HYPER_FLOATS = len(L.AdamHyper._fields_)
NORM_PARTIALS = 1024                 # workspace floats of the clip-norm reduction (kNormBlocks, csrc/loss_optim.cu)


def _check_adam(p, g, m, v, norm_out, workspace, hyper=None) -> None:
    _require_cuda(p, g, m, v, norm_out, workspace, hyper)
    flat = (p, g, m, v, norm_out, workspace) + (() if hyper is None else (hyper,))
    if any(t.dtype != torch.float32 or not t.is_contiguous() for t in flat):
        raise L.CstpError("adam_clip_step: every buffer must be contiguous fp32")
    if len({p.numel(), g.numel(), m.numel(), v.numel()}) != 1 or p.numel() == 0:
        raise L.CstpError(f"adam_clip_step: p, g, m, v need one non-zero length, got "
                          f"{[t.numel() for t in (p, g, m, v)]}")
    if norm_out.numel() < 2 or workspace.numel() < NORM_PARTIALS or (hyper is not None and hyper.numel() < ADAM_HYPER_FLOATS):
        raise L.CstpError(f"adam_clip_step: norm_out needs 2 floats, workspace {NORM_PARTIALS}, hyper {ADAM_HYPER_FLOATS}")


def adam_clip_step(p, g, m, v, hyper: tuple, norm_out, workspace) -> None:
    """clip_grad_norm_ + one Adam / AdamW step on flat fp32 buffers (p, g, exp_avg m, exp_avg_sq v); `hyper` holds the
    ten cstp_adam_hyper scalars in field order (engine.adam_scalars computes them)."""
    _check_adam(p, g, m, v, norm_out, workspace)
    L.check(L.load().cstp_adam_clip_step(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), L.AdamHyper(*map(float, hyper)),
                                         _ptr(norm_out), _ptr(workspace), _stream()))


def adam_clip_step_dev(p, g, m, v, hyper, norm_out, workspace) -> None:
    """adam_clip_step with the scalars read from the device vector `hyper` (fp32 [10]) at run time: the form a captured
    CUDA graph replays while the host rewrites the step-dependent scalars before every replay."""
    _check_adam(p, g, m, v, norm_out, workspace, hyper)
    L.check(L.load().cstp_adam_clip_step_dev(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), _ptr(hyper), _ptr(norm_out),
                                             _ptr(workspace), _stream()))


def kernel_name(plan) -> str:
    """CUDA kernel a plan object launches (for profiles and the bench roofline)."""
    inner = getattr(plan, "plan", plan)          # WgradSpec wraps its plan
    return {ConvHaloPlan: "conv_halo_kernel", ConvPlan: "conv_gemm_kernel", WgradHaloPlan: "wgrad_halo_kernel",
            WgradPlan: "wgrad_gemm_kernel"}.get(type(inner), type(inner).__name__)


_replayed_launches = 0


def note_replayed(n: int) -> None:
    """Kernel launches replayed from a captured CUDA graph (the C-side counter only sees direct launches)."""
    global _replayed_launches
    _replayed_launches += int(n)


def launch_count() -> int:
    """Kernels of this library launched so far: direct launches through the C ABI plus launches replayed from CUDA graphs."""
    return int(L.load().cstp_launch_count()) + _replayed_launches


def jpeg_workspace_bytes(width: int, height: int) -> int:
    """Workspace bytes cstp_jpeg_decode needs for one image of this size (any supported sampling)."""
    v = L.load().cstp_jpeg_workspace_bytes(int(width), int(height))
    if v < 0:
        raise ValueError(f"JPEG frame size {width}x{height} outside 1 .. 65535")
    return v


def jpeg_decode(staged, data_offset: int, n_images: int, status, workspace) -> None:
    """Decodes a batch staged in one uint8 device buffer: n_images cstp_jpeg_image descriptors at its start, the
    concatenated streams from data_offset.  status: int32 [n_images]; workspace: uint8, each image's slice at its
    descriptor's ws_offset."""
    _require_cuda(staged, status, workspace)
    if staged.dtype != torch.uint8 or status.dtype != torch.int32 or status.numel() < n_images \
            or workspace.dtype != torch.uint8 or not (staged.is_contiguous() and workspace.is_contiguous()):
        raise L.CstpError("jpeg_decode: contiguous uint8 staging and workspace buffers, int32 status [n_images]")
    base = staged.data_ptr()
    L.check(L.load().cstp_jpeg_decode(C.c_void_p(base + data_offset), C.c_void_p(base), n_images, _ptr(status),
                                      _ptr(workspace), workspace.numel(), _stream()))
