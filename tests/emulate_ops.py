"""CPU stand-in for `cstp_b200.ops` -- TEST INFRASTRUCTURE ONLY.

Implements, in plain torch on CPU tensors, exactly what each C-ABI entry point is specified to compute (same
signatures as cstp_b200.ops, same packed-weight / padded-NDHWC / flat-buffer layouts, bf16 storage rounding), so the
host-side orchestration of cstp_b200.engine (buffer wiring, program order, residual/accumulate flags, flat parameter
layout) can be validated against the oracle without a GPU.  Tests inject it with monkeypatch; nothing under
cstp_b200/ imports it and the product path has no CPU route.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from cstp_b200 import lib as L  # noqa: F401  (engine reaches CstpError through ops.L)
from cstp_b200 import ops as real
from cstp_b200.ops import (BNState, ConvGeom, pad16, pad64, fwd_taps, dgrad_classes, bn_nblocks, pick_box,  # noqa: F401
                           wgrad_partials_need, wgrad_halo_layout, STEM_GEOM, STEM_CHANNELS)

from .emulate import _gather

_launches = 0


def _count(n=1):
    global _launches
    _launches += n


def require_device(*tensors):
    pass


def launch_count():
    return _launches


def kernel_name(plan):
    return "emulated"


class _Plan:
    def __init__(self, fn):
        self.fn = fn
        self.splits = 1

    def run(self):
        _count()
        self.fn()


def _store(out, out_f32, val, accumulate):
    """val fp32 (..., Np) -> bf16 and/or fp32 outputs with the kernel's accumulate semantics."""
    if out is not None:
        if accumulate:
            val = val + out.float()
        out.copy_(val.to(out.dtype))
    if out_f32 is not None:
        if accumulate and out is None:
            val = val + out_f32
        out_f32.copy_(val)


def _prologue(x, st):
    """What the kernels' operand prologue feeds the tensor cores: relu(bn(x)) of the producer, rounded to the storage
    type, per statistics group (equal parts of the N axis)."""
    if st is None:
        return x.float()
    G, N = st.groups, x.shape[0]
    xf = x.float().reshape(G, N // G, -1, x.shape[-1])
    y = (xf * st.scale.view(G, 1, 1, -1) + st.shift.view(G, 1, 1, -1)).clamp_min(0)
    return y.reshape(x.shape).to(x.dtype).float()


def conv_fwd_plan(x, w_packed, out, geom: ConvGeom, *, out_f32=None, bias=None, accumulate=False, n_tile=None, box=None,
                  allow_halo=True, stats=None, prologue=None):       # stats: never fused here (plan.stat_blocks stays 0)
    N, T, H, W, Ca = x.shape
    To, Ho, Wo = geom.out_dims(T, H, W)
    ref = out if out is not None else out_f32
    Np = ref.shape[-1]
    Kc = pad64(Ca)
    assert tuple(ref.shape[:4]) == (N, To, Ho, Wo)
    assert w_packed.shape[0] >= Np and w_packed.shape[1] == geom.taps * Kc
    maps, taps = fwd_taps(geom)

    def run():
        acc = torch.zeros(N, To, Ho, Wo, Np)
        xf = _prologue(x, prologue)
        for (m, dw, dh, dt, ti) in taps:
            a = _gather(xf, maps[m], geom.stride, (dw, dh, dt), (Wo, Ho, To, N))
            acc += a @ w_packed[:Np, ti * Kc: ti * Kc + Ca].float().t()
        if bias is not None:
            acc += bias[:Np]
        _store(out, out_f32, acc, accumulate)
    return _Plan(run)


def conv_dgrad_plans(g, wt_packed, dx, geom: ConvGeom, *, accumulate=False):
    N, T, H, W, Ci = dx.shape
    Co = g.shape[-1]
    Kc = pad64(Co)
    assert wt_packed.shape[0] >= Ci and wt_packed.shape[1] == geom.taps * Kc
    plans, covers = [], True
    for cl in dgrad_classes(tuple(dx.shape), geom):
        if not cl["taps"]:
            covers = False
            continue

        def run(cl=cl):
            Wt, Ht, Tt, Nt = cl["space"]
            acc = torch.zeros(Nt, Tt, Ht, Wt, Ci)
            gf = g.float()
            for (dw, dh, dt, ti) in cl["taps"]:
                a = _gather(gf, (0, 0, 0), (1, 1, 1), (dw, dh, dt), cl["space"])
                acc += a @ wt_packed[:Ci, ti * Kc: ti * Kc + Co].float().t()
            ct, ch, cw = cl["cls"]
            st, sh, sw = geom.stride
            sub = dx[:, ct::st, ch::sh, cw::sw, :]
            if accumulate:
                acc = acc + sub.float()
            sub.copy_(acc.to(dx.dtype))
        plans.append(_Plan(run))
    return plans, covers


def linear_plan(x, w_packed, out, *, out_f32=None, bias=None, accumulate=False):
    B, Ca = x.shape
    ref = out if out is not None else out_f32
    Np = ref.shape[-1]
    x5 = x.view(1, 1, 1, B, Ca)
    o5 = None if out is None else out.view(1, 1, 1, B, Np)
    of5 = None if out_f32 is None else out_f32.view(1, 1, 1, B, Np)
    return conv_fwd_plan(x5, w_packed, o5, ConvGeom((1, 1, 1)), out_f32=of5, bias=bias, accumulate=accumulate)


class _WgradSpec:
    def __init__(self, x, g, geom, cout, cin, prologue=None, layout=0):
        self.x, self.g, self.geom, self.cout, self.cin, self.prologue = x, g, geom, cout, cin, prologue
        self.layout = layout
        self.plan = _Plan(lambda: None)

    def run(self, dw, accumulate=False):
        _count(2)
        x, g, geom = _prologue(self.x, self.prologue), self.g.float(), self.geom
        N, T, H, W, Ci = x.shape
        _, To, Ho, Wo, Co = g.shape
        maps, taps = fwd_taps(geom)
        res = torch.zeros(self.cout, self.cin, geom.taps)
        for (m, dw_, dh, dt, ti) in taps:
            a = _gather(x, maps[m], geom.stride, (dw_, dh, dt), (Wo, Ho, To, N))
            res[:, :, ti] = (g.reshape(-1, Co).t() @ a.reshape(-1, Ci))[:self.cout, :self.cin]
        if self.layout == 1:       # stem row pairs: res[co][hpar*32 + kw*3 + c][j] -> dW (cout, 3, 1, 7, 7), kh = 2j + hpar - 1
            r5 = res.reshape(self.cout, 2, 32, 4)[:, :, :21].reshape(self.cout, 2, 7, 3, 4)      # co, hpar, kw, c, j
            r5 = r5.permute(0, 3, 4, 1, 2).reshape(self.cout, 3, 8, 7)                           # co, c, 2j + hpar, kw
            res = r5[:, :, 1:, :]
        res = res.reshape(dw.shape)
        dw.copy_(dw + res if accumulate else res)


def wgrad_plan(x, g, geom, cout, cin, partials, *, splits=None, box=None, sms=148, prologue=None, layout=0):
    need_chunks = geom.taps * (pad64(x.shape[-1]) // 64)
    if need_chunks > L.CSTP_MAX_MCHUNKS:
        raise L.CstpError("too many M chunks")
    return _WgradSpec(x, g, geom, cout, cin, prologue, layout)


def pack_weight(w, packed, *, transpose=False):
    _count()
    cout, cin = w.shape[0], w.shape[1]
    taps = w.numel() // (cout * cin)
    Rp, Ktot = packed.shape
    if int(transpose) == 2:    # stem: packed[co][j*64 + hpar*32 + kw*3 + c] = w[co][c][0][2j + hpar - 1][kw]
        packed.zero_()
        w8 = F.pad(w.reshape(cout, 3, 7, 7), (0, 0, 1, 0))                    # kh' = kh + 1 = 2j + hpar in 0..7
        w8 = w8.reshape(cout, 3, 4, 2, 7).permute(0, 2, 3, 4, 1).reshape(cout, 4, 2, 21)      # co, j, hpar, kw*3 + c
        packed.view(Rp, 4, 2, 32)[:cout, :, :, :21] = w8.to(packed.dtype)
        return
    Kc = Ktot // taps
    w3 = w.reshape(cout, cin, taps)
    packed.zero_()
    p3 = packed.view(Rp, taps, Kc)
    if not transpose:
        p3[:cout, :, :cin] = w3.permute(0, 2, 1).to(packed.dtype)
    else:
        p3[:cin, :, :cout] = w3.permute(1, 2, 0).to(packed.dtype)


class PackList:
    def __init__(self, jobs, device):
        self.jobs = jobs

    def run(self):
        for w, packed, transpose in self.jobs:
            pack_weight(w, packed, transpose=transpose)


def stem_pack(x, P):
    _count()
    N, C, T, H, W = x.shape
    Wo = W // 2
    xp = F.pad(x, (3, 3))                                    # (N, 3, T, H, W + 6)
    taps = xp.unfold(4, 7, 2)                                # (N, 3, T, H, Wo, 7): [..., wo, kw] = x[2*wo + kw - 3]
    P.zero_()
    rows = taps.permute(0, 2, 3, 4, 5, 1).reshape(N, T, H // 2, 2, Wo, 21)          # n, t, h2, hpar, wo, kw*3 + c
    P.view(N, T, H // 2, Wo, 2, 32)[..., :21] = rows.permute(0, 1, 2, 4, 3, 5).to(P.dtype)


def _group_view(t, groups):
    rows = t.numel() // t.shape[-1]
    return t.reshape(groups, rows // groups, t.shape[-1])


def bn_forward_stats(raw, st: BNState, gamma, beta, running_mean, running_var, eps=1e-5, momentum=0.1, fused_blocks=0,
                     sync=None):
    _count(2)
    x = _group_view(raw, st.groups).float()
    n = x.shape[1]
    C, Cp = st.C, st.Cp
    s1, s2 = x.double().sum(1), (x.double() ** 2).sum(1)
    if sync is not None and sync.world > 1:          # SyncBN: one [groups][2][Cp] fp32 row summed over the ranks
        row = torch.stack([s1, s2], 1).float()
        sync.all_reduce(row)
        s1, s2, n = row[:, 0].double(), row[:, 1].double(), n * sync.world
    mean = s1 / n
    var = s2 / n - mean ** 2
    var.clamp_(min=0)
    istd = (1.0 / torch.sqrt(var + eps)).float()
    mean_f = mean.float()
    sc = torch.zeros(st.groups, Cp)
    sh = torch.zeros(st.groups, Cp)
    sc[:, :C] = gamma * istd[:, :C]
    sh[:, :C] = beta - mean_f[:, :C] * sc[:, :C]
    st.scale.copy_(sc.reshape(-1))
    st.shift.copy_(sh.reshape(-1))
    m_ = torch.zeros(st.groups, Cp)
    i_ = torch.zeros(st.groups, Cp)
    m_[:, :C], i_[:, :C] = mean_f[:, :C], istd[:, :C]
    st.mean.copy_(m_.reshape(-1))
    st.invstd.copy_(i_.reshape(-1))
    if running_mean is not None:
        for g in range(st.groups):
            unb = var[g, :C] * n / (n - 1) if n > 1 else var[g, :C]
            running_mean.copy_((1 - momentum) * running_mean + momentum * mean_f[g, :C])
            running_var.copy_((1 - momentum) * running_var + momentum * unb.float())


def bn_apply(raw, st: BNState, out, *, relu, res=None, res_state=None, res_relu=False):
    _count()
    x = _group_view(raw, st.groups).float()
    y = x * st.scale.view(st.groups, 1, -1) + st.shift.view(st.groups, 1, -1)
    if res is not None:
        r = _group_view(res, st.groups).float()
        if res_state is not None:
            r = r * res_state.scale.view(st.groups, 1, -1) + res_state.shift.view(st.groups, 1, -1)
            if res_relu:
                r = r.clamp_min(0).to(res.dtype).float()
        y = y + r
    if relu:
        y = y.clamp_min(0)
    out.copy_(y.reshape(out.shape).to(out.dtype))


def bn_backward(d, act, raw, st: BNState, gamma, dgamma, dbeta, g_out, *, dz=None, accumulate=False,
                mask_from_raw=False, sync=None):
    _count(3)
    G, C, Cp = st.groups, st.C, st.Cp
    dy = _group_view(d, G).float()
    if mask_from_raw:
        # the very expression bn_apply evaluated in the forward pass (the kernels use the same fmaf in both places)
        pre = _group_view(raw, G).float() * st.scale.view(G, 1, Cp) + st.shift.view(G, 1, Cp)
        dy = dy * (pre > 0)
    elif act is not None:
        dy = dy * (_group_view(act, G).float() > 0)
    if dz is not None:
        dz.copy_(dy.reshape(dz.shape).to(dz.dtype))
    x = _group_view(raw, G).float()
    n = x.shape[1]
    xhat = (x - st.mean.view(G, 1, Cp)) * st.invstd.view(G, 1, Cp)
    s = dy.double().sum(1)
    sx = (dy * xhat).double().sum(1)
    s_loc, sx_loc = s, sx                              # dgamma / dbeta stay local sums under SyncBN
    if sync is not None and sync.world > 1:
        row = torch.stack([s, sx], 1).float()
        sync.all_reduce(row)
        s, sx, n = row[:, 0].double(), row[:, 1].double(), n * sync.world
    c0 = torch.zeros(G, Cp)
    c0[:, :C] = gamma * st.invstd.view(G, Cp)[:, :C]
    c1 = (s / n).float()
    c2 = (sx / n).float()
    c1[:, C:] = 0
    c2[:, C:] = 0
    go = c0.view(G, 1, Cp) * (dy - c1.view(G, 1, Cp) - xhat * c2.view(G, 1, Cp))
    g_out.copy_(go.reshape(g_out.shape).to(g_out.dtype))
    if dgamma is not None:
        dg, db = sx_loc.sum(0)[:C].float(), s_loc.sum(0)[:C].float()
        dgamma.copy_(dgamma + dg if accumulate else dg)
        dbeta.copy_(dbeta + db if accumulate else db)


def avgpool_fwd(x, out_f32, out_bf16, rows_out=None, ld_out=None):
    _count()
    N, Cp = x.shape[0], x.shape[-1]
    m = x.float().reshape(N, -1, Cp).mean(1)
    rows_out = rows_out or N
    for o in (out_f32, out_bf16):
        if o is None:
            continue
        for n in range(N):
            o[n % rows_out, (n // rows_out) * Cp:(n // rows_out + 1) * Cp] = m[n].to(o.dtype)


def avgpool_bwd(dfeat, dx, dcat=None):
    _count()
    N, Cp = dx.shape[0], dx.shape[-1]
    P = dx.numel() // (N * Cp)
    v = dfeat.clone()
    if dcat is not None:
        rows_cat = dcat.shape[0]
        for n in range(N):
            v[n] += dcat[n % rows_cat, (n // rows_cat) * Cp:(n // rows_cat + 1) * Cp]
    v = v / P
    dx.copy_(v.view(N, *([1] * (dx.dim() - 2)), Cp).expand(dx.shape).to(dx.dtype))


def colsum(x, C_, out, accumulate=False):
    _count()
    s = x[:, :C_].float().sum(0)
    out.copy_(out + s if accumulate else s)


def cast_pad(x, out, cols=None, scale_dev=None):
    _count()
    cols = cols or x.shape[1]
    s = 1.0 if scale_dev is None else scale_dev.reshape(-1)[0]
    out.zero_()
    out[:, :cols] = (x[:, :cols] * s).to(out.dtype)


def byol_loss(pred, tproj, B, D, loss_out, upstream=None, dpred=None):
    _count()
    p = pred[:, :D].detach().clone().requires_grad_(True)
    t = tproj[:, :D]
    with torch.enable_grad():
        def lf(x, y):
            return 2 - 2 * (F.normalize(x, dim=-1) * F.normalize(y, dim=-1)).sum(-1)
        loss = (lf(p[:B], t[B:]) + lf(p[B:], t[:B])).mean()
        up = 1.0 if upstream is None else upstream.reshape(-1)[0]
        (gr,) = torch.autograd.grad(loss * up, p)
    loss_out.copy_(loss.detach().reshape(loss_out.shape))
    if dpred is not None:
        dpred.zero_()
        dpred[:, :D] = gr


def pretext_ce(logits, labels, dlogits, B, n_cls, weights5, losses_out):
    _count()
    w = [weights5[1], weights5[2], weights5[3], weights5[3], weights5[4], weights5[4]]
    tot = 0.0
    for h in range(6):
        lg = logits[h][:, :n_cls].detach().clone().requires_grad_(True)
        with torch.enable_grad():
            ce = F.cross_entropy(lg, labels[h])
            (gr,) = torch.autograd.grad(ce * w[h], lg)
        losses_out[h] = ce.detach()
        tot = tot + w[h] * ce.detach()
        if dlogits is not None and dlogits[h] is not None:
            dlogits[h].zero_()
            dlogits[h][:, :n_cls] = gr
    losses_out[6] = tot


def ntxent_workspace_floats(rows, d):
    return 16


def ntxent(z, temperature, use_cosine, loss_out, dz, workspace):
    _count()
    zr = z.detach().clone().requires_grad_(True)
    rows = z.shape[0]
    with torch.enable_grad():
        zn = zr / zr.norm(dim=1, keepdim=True).clamp_min(1e-8) if use_cosine else zr
        S = zn @ zn.t() / temperature
        idx = torch.arange(rows)
        pos = (idx + rows // 2) % rows
        Sm = S.masked_fill(torch.eye(rows, dtype=torch.bool), float("-inf"))
        loss = (torch.logsumexp(Sm, 1) - S[idx, pos]).mean()
        if dz is not None:
            (gr,) = torch.autograd.grad(loss, zr)
            dz.copy_(gr)
    loss_out.copy_(loss.detach().reshape(loss_out.shape))


def l2norm_fwd(x, y_bf16, norms, d, eps=1e-12):
    _count()
    n = x[:, :d].norm(dim=1).clamp_min(eps)
    y_bf16.zero_()
    y_bf16[:, :d] = (x[:, :d] / n[:, None]).to(y_bf16.dtype)
    norms.copy_(n)


def l2norm_bwd(x, norms, g_bf16, dx, d):
    _count()
    g = g_bf16[:, :d].float()
    y = x[:, :d] / norms[:, None]
    dx.zero_()
    dx[:, :d] = (g - y * (y * g).sum(1, keepdim=True)) / norms[:, None]


def ce_loss(logits, labels, n_cls, loss_out, dlogits, workspace):
    _count()
    lg = logits[:, :n_cls].detach().clone().requires_grad_(True)
    with torch.enable_grad():
        ce = F.cross_entropy(lg, labels)
        (gr,) = torch.autograd.grad(ce, lg)
    loss_out.copy_(ce.detach().reshape(loss_out.shape))
    if dlogits is not None:
        dlogits.zero_()
        dlogits[:, :n_cls] = gr


def bn_eval_coeffs(st, gamma, beta, running_mean, running_var, eps=1e-5):
    _count()
    sc = torch.zeros(st.groups, st.Cp)
    sh = torch.zeros(st.groups, st.Cp)
    s_ = gamma / torch.sqrt(running_var + eps)
    sc[:, :st.C] = s_
    sh[:, :st.C] = beta - running_mean * s_
    st.scale.copy_(sc.reshape(-1))
    st.shift.copy_(sh.reshape(-1))


def ema_update(k, q, m):
    _count()
    import numpy as np
    mf, omf = float(np.float32(m)), float(np.float32(1.0 - m))
    k.copy_(k * mf + q * omf)


def sgd_clip_step_dev(p, g, mom, hyper, norm_out, workspace):
    lr, momentum, wd, max_norm, do_clip, first = [float(v) for v in hyper.tolist()]
    sgd_clip_step(p, g, mom, lr, momentum, wd, max_norm, bool(do_clip), bool(first), norm_out, workspace)


def note_replayed(n):
    _count(n)


def sgd_clip_step(p, g, mom, lr, momentum, wd, max_norm, do_clip, first_step, norm_out, workspace):
    _count(2)
    total = g.double().pow(2).sum().sqrt().float()
    coef = torch.clamp(max_norm / (total + 1e-6), max=1.0) if do_clip else torch.tensor(1.0)
    gr = g * coef + wd * p
    b = gr if first_step else momentum * mom + gr
    mom.copy_(b)
    p.copy_(p - lr * b)
    norm_out[0], norm_out[1] = total, coef
