"""Host-side implicit-GEMM geometry (tap lists, stride-parity views, dgrad classes, wgrad chunks, tile boxes) checked
against torch's convolution functions through the descriptor interpreter in tests/emulate.py.  CPU only."""
import math

import pytest
import torch
import torch.nn.functional as F

from cstp_b200 import ops
from cstp_b200.ops import ConvGeom, fwd_taps
from tests import emulate as E

CASES = [
    # kernel, stride, pad, (N, T, H, W)  -- every conv geometry of R2Plus1DNet plus degenerate extents
    ((1, 3, 3), (1, 1, 1), (0, 1, 1), (2, 3, 8, 8)),
    ((1, 3, 3), (1, 2, 2), (0, 1, 1), (2, 2, 8, 8)),
    ((1, 3, 3), (1, 2, 2), (0, 1, 1), (1, 1, 7, 7)),
    ((3, 1, 1), (1, 1, 1), (1, 0, 0), (2, 4, 3, 3)),
    ((3, 1, 1), (2, 1, 1), (1, 0, 0), (2, 4, 4, 4)),
    ((3, 1, 1), (2, 1, 1), (1, 0, 0), (2, 1, 4, 4)),
    ((1, 1, 1), (1, 2, 2), (0, 0, 0), (2, 2, 8, 8)),
    ((1, 1, 1), (2, 1, 1), (0, 0, 0), (2, 4, 4, 4)),
    ((1, 1, 1), (1, 1, 1), (0, 0, 0), (1, 1, 1, 9)),
]


@pytest.mark.parametrize("k,s,p,shape", CASES)
def test_descriptor_semantics_match_torch(k, s, p, shape):
    torch.manual_seed(0)
    N, T, H, W = shape
    g = ConvGeom(k, s, p)
    ci, co = 5, 7
    x = torch.randn(N, T, H, W, ci)
    w = torch.randn(co, ci, *k)
    xr = x.permute(0, 4, 1, 2, 3)
    ref = F.conv3d(xr, w, stride=s, padding=p).permute(0, 2, 3, 4, 1)
    assert tuple(ref.shape[1:4]) == g.out_dims(T, H, W)
    torch.testing.assert_close(E.emulate_fwd(x, w, g), ref, rtol=1e-4, atol=1e-4)
    gg = torch.randn_like(ref)
    gr = gg.permute(0, 4, 1, 2, 3)
    dref = torch.nn.grad.conv3d_input((N, ci, T, H, W), w, gr, stride=s, padding=p).permute(0, 2, 3, 4, 1)
    dx, covers = E.emulate_dgrad(gg, w, g, (N, T, H, W, ci))
    torch.testing.assert_close(dx, dref, rtol=1e-4, atol=1e-4)
    # a class without taps exists exactly when some input position is never read by the conv
    never_read = any(all((c + pp - a) % st != 0 for a in range(kk)) for kk, st, pp, ext in zip(k, s, p, (T, H, W))
                     for c in range(min(st, ext)))
    assert covers == (not never_read)
    wref = torch.nn.grad.conv3d_weight(xr, w.shape, gr, stride=s, padding=p)
    torch.testing.assert_close(E.emulate_wgrad(x, gg, g, co, ci), wref, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("space,rows", [((56, 56, 16, 120), 128), ((7, 7, 2, 8), 128), ((1, 1, 1, 60), 128),
                                        ((28, 28, 8, 3), 64), ((14, 14, 4, 1), 64), ((6021120, 1, 1, 1), 128)])
def test_pick_box(space, rows):
    bw, bh, bt, bn = ops.pick_box(*space, rows)
    assert bw * bh * bt * bn == rows and max(bw, bh, bt, bn) <= 256
    tiles = math.prod(math.ceil(d / b) for d, b in zip(space, (bw, bh, bt, bn)))
    # never worse than the trivial row-major box
    trivial = math.ceil(space[0] / rows) * space[1] * space[2] * space[3]
    assert tiles <= trivial


def test_view5_geometry_matches_strided_slicing():
    x = torch.arange(2 * 5 * 6 * 7 * 16).view(2, 5, 6, 7, 16)
    for parity, stride in [((0, 0, 0), (1, 1, 1)), ((1, 0, 1), (2, 1, 2)), ((0, 1, 1), (1, 2, 2)), ((1, 1, 1), (2, 2, 2))]:
        off, dims, strides = ops.view5_geometry(tuple(x.shape), parity, stride)
        sub = x[:, parity[0]::stride[0], parity[1]::stride[1], parity[2]::stride[2], :]
        assert dims == (16, sub.shape[3], sub.shape[2], sub.shape[1], sub.shape[0])
        v = torch.as_strided(x.reshape(-1), (dims[4], dims[3], dims[2], dims[1], dims[0]),
                             (strides[3], strides[2], strides[1], strides[0], 1), off)
        assert torch.equal(v, sub)


def test_intermediate_channels_table():
    """SURVEY.md A.1 / r21d_byol.py:74-76: the odd mid-channel counts of every factorised conv."""
    from cstp_b200.engine import intermed_channels as ic
    assert ic(3, 64, (3, 7, 7)) == 83
    assert [ic(64, 64, (3, 3, 3)), ic(64, 128, (3, 3, 3)), ic(128, 128, (3, 3, 3))] == [144, 230, 288]
    assert [ic(128, 256, (3, 3, 3)), ic(256, 256, (3, 3, 3)), ic(256, 512, (3, 3, 3)), ic(512, 512, (3, 3, 3))] == [460, 576, 921, 1152]
    assert [ic(64, 128, (1, 1, 1)), ic(128, 256, (1, 1, 1)), ic(256, 512, (1, 1, 1))] == [42, 85, 170]


@pytest.mark.parametrize("k,p,shape,cin,cout", [
    ((1, 3, 3), (0, 1, 1), (2, 3, 16, 24), 64, 144),      # conv2 spatial (two N tiles)
    ((3, 1, 1), (1, 0, 0), (1, 8, 8, 16), 144, 64),       # conv2 temporal (3 channel chunks, last one 16 wide)
    ((3, 1, 1), (1, 0, 0), (2, 4, 6, 8), 83, 64),         # stem temporal, ragged tiles
    ((1, 3, 3), (0, 1, 1), (1, 2, 10, 12), 128, 32),
    ((1, 3, 3), (0, 1, 1), (1, 1, 16, 24), 128, 240),     # 2-D halo, two channel chunks, 5 N tiles (conv3.conv2.spatial)
])
def test_wgrad_halo_layout_semantics(k, p, shape, cin, cout):
    """Interprets ops.wgrad_halo_layout exactly as csrc/wgrad_halo.cu does (staged X boxes with halo, chunks as row
    shifts, zero OOB fill, chunk -> (tap, channel) scatter of cstp_wgrad_finalize) and compares with torch's wgrad."""
    import torch.nn.functional as F  # noqa: F401
    from cstp_b200.ops import wgrad_halo_layout, pad16
    N, T, H, W = shape
    geom = ConvGeom(k, (1, 1, 1), p)
    Ca, Np = pad16(cin), pad16(cout)
    g_ = torch.Generator().manual_seed(3)
    x = torch.zeros(N, T, H, W, Ca)
    x[..., :cin] = torch.randn(N, T, H, W, cin, generator=g_)
    gr = torch.zeros(N, T, H, W, Np)
    gr[..., :cout] = torch.randn(N, T, H, W, cout, generator=g_)
    lay = wgrad_halo_layout(tuple(x.shape), tuple(gr.shape), geom)
    assert lay is not None
    bw, bh, bt, bn = lay["box"]
    hw, hh, ht = lay["halo"]
    pitch = lay["pitch"]                    # box rows between the 8-position atoms of a chunk (8: contiguous rows)
    assert all(off % (1024 if pitch == 8 else 128) == 0 for off, _, _ in lay["chunks"])
    box_rows = lay["xbox_bytes"] // 128      # staged boxes start on 1024-byte boundaries
    offs = [c[0] for c in lay["chunks"]]
    assert all(offs[i] < offs[i + 1] for i in range(len(offs) - 1))

    def fetch(t, c0, w0, h0, t0, n0, ew, eh, et):
        """TMA box (64 ch, ew, eh, et, 1) at the given origin with zero fill outside the tensor -> [rows][64]."""
        out = torch.zeros(et, eh, ew, 64)
        for a in range(et):
            for b in range(eh):
                for c in range(ew):
                    tt, hh_, ww = t0 + a, h0 + b, w0 + c
                    if 0 <= tt < t.shape[1] and 0 <= hh_ < t.shape[2] and 0 <= ww < t.shape[3] and n0 < t.shape[0]:
                        ce = min(64, t.shape[-1] - c0)
                        if ce > 0:
                            out[a, b, c, :ce] = t[n0, tt, hh_, ww, c0:c0 + ce]
        return out.reshape(-1, 64)

    # `flip`: the taps ride on dL/d(raw) (M = (tap, cout chunk)) and the activations are the N side (columns = cin)
    flip = lay["flip"]
    m_side, n_side = (gr, x) if flip else (x, gr)
    n_cols = Ca if flip else Np
    n_chunks = len(lay["chunks"])
    P = torch.zeros(n_chunks * 64, n_cols)
    for n0 in range(N):
        for t0 in range(0, T, bt):
            for h0 in range(0, H, bh):
                for w0 in range(0, W, bw):
                    boxes = [fetch(m_side, c0, w0 + dw, h0 + dh, t0 + dt, n0, bw + hw, bh + hh, bt + ht)
                             for (c0, dw, dh, dt) in lay["xboxes"]]
                    staged = torch.cat([torch.cat([b_, torch.zeros(box_rows - b_.shape[0], 64)], 0) for b_ in boxes], 0)
                    G = torch.cat([fetch(n_side, c0, w0, h0, t0, n0, bw, bh, bt) for c0 in range(0, n_cols, 64)], 1)[:, :n_cols]
                    for i, (off, _, _) in enumerate(lay["chunks"]):
                        idx = [off // 128 + a_ * pitch + j for a_ in range(8) for j in range(8)]
                        rows = staged[idx]
                        P[i * 64:(i + 1) * 64] += rows.t() @ G
    dw_ = torch.zeros(cout, cin, geom.taps)
    for i, (_, tap, c0) in enumerate(lay["chunks"]):
        for r in range(64):
            if flip and c0 + r < cout:
                dw_[c0 + r, :, tap] = P[i * 64 + r, :cin]
            elif not flip and c0 + r < cin:
                dw_[:, c0 + r, tap] = P[i * 64 + r, :cout]
    ref = torch.nn.grad.conv3d_weight(x[..., :cin].permute(0, 4, 1, 2, 3), (cout, cin, *k),
                                      gr[..., :cout].permute(0, 4, 1, 2, 3), stride=1, padding=p)
    assert torch.allclose(dw_.reshape(ref.shape), ref, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("k,p,shape,cin,cout,dgrad", [
    ((1, 3, 3), (0, 1, 1), (2, 2, 20, 12), 64, 144, False),
    ((3, 1, 1), (1, 0, 0), (1, 20, 8, 8), 144, 64, False),
    ((1, 3, 3), (0, 1, 1), (1, 1, 18, 40), 144, 64, True),
    ((3, 1, 1), (1, 0, 0), (2, 5, 4, 12), 64, 144, True),
    ((1, 3, 3), (0, 1, 1), (1, 2, 32, 16), 64, 144, False),     # 2-D halo (8 x 16 tiles, one box for nine taps)
    ((1, 3, 3), (0, 1, 1), (1, 1, 16, 24), 144, 64, True),      # 2-D halo dgrad with a 16-channel tail
])
def test_conv_halo_layout_semantics(k, p, shape, cin, cout, dgrad):
    """Interprets ops.conv_halo_layout exactly as csrc/conv_halo.cu does (one staged halo box per load group and
    channel chunk, taps as row shifts, zero OOB fill) and compares with torch conv3d / its input gradient."""
    import torch.nn.functional as F
    from cstp_b200.ops import conv_halo_layout, dgrad_classes, pad16, pad64
    N, T, H, W = shape
    geom = ConvGeom(k, (1, 1, 1), p)
    gen = torch.Generator().manual_seed(5)
    w = torch.randn(cout, cin, *k, generator=gen)
    if not dgrad:
        a_c, n_c = cin, cout
        _, taps = fwd_taps(geom)
        taps = [(dw, dh, dt, ti) for (_, dw, dh, dt, ti) in taps]
        wmat = lambda ti: w.reshape(cout, cin, -1)[:, :, ti]                     # [n][c]   # noqa: E731
    else:
        a_c, n_c = cout, cin
        (cl,) = dgrad_classes((N, T, H, W, pad16(cin)), geom)
        taps = cl["taps"]
        wmat = lambda ti: w.reshape(cout, cin, -1)[:, :, ti].t()                 # [n = ci][c = co]  # noqa: E731
    Ca, Np = pad16(a_c), pad16(n_c)
    a = torch.zeros(N, T, H, W, Ca)
    a[..., :a_c] = torch.randn(N, T, H, W, a_c, generator=gen)
    lay = conv_halo_layout((W, H, T, N), [(dw, dh, dt, ti * pad64(Ca)) for (dw, dh, dt, ti) in taps], Ca, Np)
    assert lay is not None
    bw, bh, bt, bn = lay["box"]
    hw, hh, ht = lay["halo"]
    pitch = lay["pitch"]                    # box rows between the 8-row atoms of a tap (8: its 128 rows are contiguous)
    assert bw * bh * bt * bn == 128 and all(s_ % (1024 if pitch == 8 else 128) == 0 for s_, _ in lay["taps"])
    out = torch.zeros(N, T, H, W, n_c)
    tap_of_koff = {ti * pad64(Ca): ti for (_, _, _, ti) in taps}

    def fetch(c0, w0, h0, t0, n0):
        box = torch.zeros(bt + ht, bh + hh, bw + hw, 64)
        for aa in range(bt + ht):
            for bb in range(bh + hh):
                for cc in range(bw + hw):
                    tt, hh_, ww = t0 + aa, h0 + bb, w0 + cc
                    if 0 <= tt < T and 0 <= hh_ < H and 0 <= ww < W:
                        ce = min(64, Ca - c0)
                        box[aa, bb, cc, :ce] = a[n0, tt, hh_, ww, c0:c0 + ce]
        return box.reshape(-1, 64)

    for n0 in range(N):
        for t0 in range(0, T, bt):
            for h0 in range(0, H, bh):
                for w0 in range(0, W, bw):
                    acc = torch.zeros(128, n_c)
                    for (gdw, gdh, gdt, first, cnt) in lay["groups"]:
                        for c0 in range(0, Ca, 64):
                            staged = fetch(c0, w0 + gdw, h0 + gdh, t0 + gdt, n0)
                            for (shift, k_off) in lay["taps"][first:first + cnt]:
                                rows = staged[[shift // 128 + a_ * pitch + j for a_ in range(16) for j in range(8)]]
                                wm = wmat(tap_of_koff[k_off])[:, c0:c0 + 64]
                                acc += rows[:, :wm.shape[1]] @ wm.t()
                    for r in range(128):
                        ww, hh_, tt = w0 + r % bw, h0 + (r // bw) % bh, t0 + r // (bw * bh)
                        if ww < W and hh_ < H and tt < T:
                            out[n0, tt, hh_, ww] = acc[r]
    x5 = a[..., :a_c].permute(0, 4, 1, 2, 3)
    if not dgrad:
        ref = F.conv3d(x5, w, None, 1, p)
    else:
        ref = torch.nn.grad.conv3d_input((N, cin, T, H, W), w, x5, stride=1, padding=p)
    assert torch.allclose(out.permute(0, 4, 1, 2, 3), ref, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("k,p,shape,cin,cout,dgrad,G", [
    ((1, 3, 3), (0, 1, 1), (1, 2, 12, 12), 64, 144, True, 4),      # dgrad of the 64 -> 144 1x3x3 layers (conv2.*.spatial): slab axis h
    ((1, 3, 3), (0, 1, 1), (2, 3, 10, 20), 64, 144, True, 4),      # partial slab group along h, partial tiles along w / t
    ((1, 3, 3), (0, 1, 1), (2, 3, 7, 20), 64, 80, True, 2),        # two rows per tile, 16-channel tail of the operand, odd H
    ((1, 3, 3), (0, 1, 1), (1, 2, 11, 12), 64, 96, True, 3),       # three rows per tile (ragged last group), 32-channel tail
    ((1, 3, 3), (0, 1, 1), (1, 1, 9, 8), 64, 64, False, 3),        # forward-shaped tap list (the kernel takes either)
])
def test_conv_slab_layout_semantics(k, p, shape, cin, cout, dgrad, G):
    """Interprets ops.conv_slab_layout + ops.slab_tables exactly as csrc/conv_halo.cu's slab mode does: every input slab
    of a tile is staged once (w halo box, zero OOB fill) and multiplied, per w tap, with `width` stacked weight rows
    starting at `brow` into the accumulator columns `doff`..; the slabs flagged `init` overwrite.  Compared with torch
    conv3d / its input gradient."""
    import torch.nn.functional as F
    from cstp_b200.ops import conv_slab_layout, slab_tables, dgrad_classes, pad16, pad64
    N, T, H, W = shape
    geom = ConvGeom(k, (1, 1, 1), p)
    gen = torch.Generator().manual_seed(7)
    w = torch.randn(cout, cin, *k, generator=gen)
    if not dgrad:
        a_c, n_c = cin, cout
        _, taps = fwd_taps(geom)
        taps = [(dw, dh, dt, ti) for (_, dw, dh, dt, ti) in taps]
        wmat = lambda ti: w.reshape(cout, cin, -1)[:, :, ti]                     # [n][c]   # noqa: E731
    else:
        a_c, n_c = cout, cin
        (cl,) = dgrad_classes((N, T, H, W, pad16(cin)), geom)
        taps = cl["taps"]
        wmat = lambda ti: w.reshape(cout, cin, -1)[:, :, ti].t()                 # [n = ci][c = co]  # noqa: E731
    Ca, Np = pad16(a_c), pad16(n_c)
    assert Np == 64
    a = torch.zeros(N, T, H, W, Ca)
    a[..., :a_c] = torch.randn(N, T, H, W, a_c, generator=gen)
    lay = conv_slab_layout((W, H, T, N), [(dw, dh, dt, ti * pad64(Ca)) for (dw, dh, dt, ti) in taps], Ca, Np, G)
    assert lay is not None and lay["slabs"][0] == G
    _, axis, nslots = lay["slabs"]
    bw, bh, bt, bn = lay["box"]
    hw = lay["halo"][0]
    pitch = lay["pitch"]
    assert axis == 1 and bw * bh * bt * bn == 128 and bh == 1 and lay["n_tile"] == G * Np
    (gdw, gdh, gdt, _, _), = lay["groups"]
    tap_of_koff = {ti * pad64(Ca): ti for (_, _, _, ti) in taps}
    nw = len(lay["taps"]) // nslots
    # stacked weight block of w tap j: [nslots * Np rows][Ca]
    stack = [torch.cat([torch.nn.functional.pad(wmat(tap_of_koff[lay["taps"][j * nslots + sl][1]]), (0, Ca - a_c, 0, Np - n_c))
                        for sl in range(nslots)]) for j in range(nw)]
    assert all(lay["taps"][j * nslots + sl][0] == j * 128 * (1 if hw else 0) for j in range(nw) for sl in range(nslots))
    table = slab_tables(G, nslots, Np)

    def fetch(w0, h0, t0, n0):          # the staged box: rows (n, t, h, w) with w fastest, bw + hw wide
        box = torch.zeros(bn, bt, bh, bw + hw, Ca)
        for nn in range(bn):
            for aa in range(bt):
                for bb in range(bh):
                    for cc in range(bw + hw):
                        n_, tt, hh_, ww = n0 + nn, t0 + aa, h0 + bb, w0 + cc
                        if n_ < N and 0 <= tt < T and 0 <= hh_ < H and 0 <= ww < W:
                            box[nn, aa, bb, cc] = a[n_, tt, hh_, ww]
        return box.reshape(-1, Ca)

    out = torch.zeros(N, T, H, W, n_c)
    for n0 in range(0, N, bn):
        for t0 in range(0, T, bt):
            for h0 in range(0, H, G):
                for w0 in range(0, W, bw):
                    acc = torch.full((128, G * Np), float("nan"))        # stale accumulator: the init slabs must overwrite
                    for (s, init, doff, brow, width) in table:
                        staged = fetch(w0 + gdw, h0 + gdh + s, t0 + gdt, n0)
                        first = init
                        for j in range(nw):
                            rows = staged[[j + a_ * pitch + r for a_ in range(16) for r in range(8)]]
                            prod = rows @ stack[j][brow:brow + width].t()
                            acc[:, doff:doff + width] = prod if first else acc[:, doff:doff + width] + prod
                            first = False
                    assert not torch.isnan(acc).any()
                    for r in range(128):
                        ww, hh_, tt, n_ = w0 + r % bw, h0 + (r // bw) % bh, t0 + (r // (bw * bh)) % bt, n0 + r // (bw * bh * bt)
                        for o in range(G):
                            if ww < W and n_ < N and hh_ + o < H and tt < T:
                                out[n_, tt, hh_ + o, ww] = acc[r, o * Np:o * Np + n_c]
    x5 = a[..., :a_c].permute(0, 4, 1, 2, 3)
    if not dgrad:
        ref = F.conv3d(x5, w, None, 1, p)
    else:
        ref = torch.nn.grad.conv3d_input((N, cin, T, H, W), w, x5, stride=1, padding=p)
    assert torch.allclose(out.permute(0, 4, 1, 2, 3), ref, rtol=1e-4, atol=1e-3)


def test_wgrad_gemm_shape_keeps_the_split_factor_behind_the_prologue():
    """csrc/wgrad.cu behind the operand prologue runs one M tile per CTA, but with the plain kernel's N tile and split-K
    factor: the same K ranges are summed in the same order, so a fused conv -> BN -> ReLU -> conv edge stays bit-identical
    to cstp_bn_apply followed by the plain kernel (tests/test_gpu_config3.py checks the bits on the GPU)."""
    for nch in (1, 2, 4, 9, 18, 27, 36, 72):
        for Np in (64, 128, 144, 256, 288, 512, 576, 1152):
            for kblocks in (4, 49, 368, 1470, 5880):
                plain = ops._wgrad_gemm_shape(nch, Np, kblocks, 148, False)
                fused = ops._wgrad_gemm_shape(nch, Np, kblocks, 148, True)
                assert fused[0] == plain[0] and fused[2] == plain[2], (nch, Np, kblocks, plain, fused)
                assert fused[1] == 1 and 1 <= plain[1] <= 4 and plain[1] * plain[0] <= 512
                assert 1 <= plain[2] <= max(1, kblocks // 4)


def test_library_is_not_stale_after_build():
    """lib.load() rebuilds when the sources changed since the library was built here (build.is_stale), never silently loads
    an old one; a fresh build is not stale."""
    from cstp_b200 import build
    build.build()
    assert build.LIB_PATH.exists() and not build.is_stale()
