"""Bring-up harness: runs each CUDA kernel family against torch fp32 references, one subprocess per case so a
device fault in one case cannot poison the others.  Usage (on a GPU box):

    python tools/gpu_kernel_check.py [case ...] > gpurun_out/kernel_check.log

This is a development tool; the graded parity tests live in tests/.
"""
from __future__ import annotations

import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _rel(a, b):
    import torch
    a, b = a.float(), b.float()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def _mk_act(N, T, H, W, C, Cp, seed):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.zeros(N, T, H, W, Cp, device="cuda", dtype=torch.bfloat16)
    x[..., :C] = torch.randn(N, T, H, W, C, device="cuda", generator=g).to(torch.bfloat16)
    return x


def case_conv(N, T, H, W, cin, cout, kernel, stride, pad, check_dgrad=True, check_wgrad=True, bias=False):
    import torch
    import torch.nn.functional as F
    from cstp_b200 import ops

    geom = ops.ConvGeom(tuple(kernel), tuple(stride), tuple(pad))
    Cip, Cop = ops.pad16(cin), ops.pad16(cout)
    x = _mk_act(N, T, H, W, cin, Cip, 1)
    gen = torch.Generator(device="cuda").manual_seed(2)
    w = torch.randn(cout, cin, *kernel, device="cuda", generator=gen) / (cin * geom.taps) ** 0.5
    wp = torch.empty(Cop, geom.taps * ops.pad64(Cip), device="cuda", dtype=torch.bfloat16)
    ops.pack_weight(w, wp)
    To, Ho, Wo = geom.out_dims(T, H, W)
    out = torch.full((N, To, Ho, Wo, Cop), float("nan"), device="cuda", dtype=torch.bfloat16)
    b = torch.randn(Cop, device="cuda") if bias else None
    plan = ops.conv_fwd_plan(x, wp, out, geom, bias=b)
    plan.run()
    torch.cuda.synchronize()
    xr = x[..., :cin].float().permute(0, 4, 1, 2, 3)
    wr = w.to(torch.bfloat16).float()
    ref = F.conv3d(xr, wr, bias=None if b is None else b[:cout], stride=stride, padding=pad).permute(0, 2, 3, 4, 1)
    res = {"fwd_cluster": getattr(plan, "cluster", 0), "fwd_rel": _rel(out[..., :cout], ref), "fwd_pad_zero": bool((out[..., cout:].float() == 0).all().item()) if not bias else True,
           "fwd_nan": int(torch.isnan(out.float()).sum().item())}
    # timing
    for _ in range(3):
        plan.run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        plan.run()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    flops = 2.0 * N * To * Ho * Wo * cout * cin * geom.taps
    res["fwd_ms"] = ms
    res["fwd_tflops"] = flops / ms / 1e9
    if check_dgrad:
        g = _mk_act(N, To, Ho, Wo, cout, Cop, 3)
        wtp = torch.empty(Cip, geom.taps * ops.pad64(Cop), device="cuda", dtype=torch.bfloat16)
        ops.pack_weight(w, wtp, transpose=True)
        dx = torch.full((N, T, H, W, Cip), float("nan"), device="cuda", dtype=torch.bfloat16)
        plans, covers = ops.conv_dgrad_plans(g, wtp, dx, geom)
        if not covers:
            dx.zero_()
        for p in plans:
            p.run()
        torch.cuda.synchronize()
        gr = g[..., :cout].float().permute(0, 4, 1, 2, 3)
        dref = torch.nn.grad.conv3d_input((N, cin, T, H, W), wr, gr, stride=stride, padding=pad).permute(0, 2, 3, 4, 1)
        res["dgrad_rel"] = _rel(dx[..., :cin], dref)
        res["dgrad_nan"] = int(torch.isnan(dx.float()).sum().item())
        res["dgrad_plans"] = len(plans)
        res["dgrad_cluster"] = max(getattr(p, "cluster", 0) for p in plans)
        e0.record()
        for _ in range(5):
            for p in plans:
                p.run()
        e1.record()
        torch.cuda.synchronize()
        res["dgrad_ms"] = e0.elapsed_time(e1) / 5
    if check_wgrad:
        g = _mk_act(N, To, Ho, Wo, cout, Cop, 3)
        part = torch.empty(64 * 1024 * 1024, device="cuda", dtype=torch.float32)
        spec = ops.wgrad_plan(x, g, geom, cout, cin, part)
        dw = torch.full_like(w, float("nan"))
        spec.run(dw)
        torch.cuda.synchronize()
        gr = g[..., :cout].float().permute(0, 4, 1, 2, 3)
        wref = torch.nn.grad.conv3d_weight(xr, w.shape, gr, stride=stride, padding=pad)
        res["wgrad_rel"] = _rel(dw, wref)
        res["wgrad_nan"] = int(torch.isnan(dw).sum().item())
        res["wgrad_splits"] = spec.plan.splits
        e0.record()
        for _ in range(5):
            spec.run(dw)
        e1.record()
        torch.cuda.synchronize()
        res["wgrad_ms"] = e0.elapsed_time(e1) / 5
        res["wgrad_tflops"] = flops / res["wgrad_ms"] / 1e9
    return res


def case_prologue(N, T, H, W, cin, cout, kernel, stride, pad, with_stats=False, iters=10):
    """Operand prologue (cstp_prologue): conv forward and weight gradient reading the producer's RAW output and applying
    its BatchNorm affine + ReLU in shared memory, against the two-pass path (cstp_bn_apply, then the plain kernels).
    Both feed the tensor cores the same bf16 values in the same order, so outputs must be bit-identical."""
    import torch
    from cstp_b200 import ops

    geom = ops.ConvGeom(tuple(kernel), tuple(stride), tuple(pad))
    Cip, Cop = ops.pad16(cin), ops.pad16(cout)
    raw = _mk_act(N, T, H, W, cin, Cip, 1)
    gen = torch.Generator(device="cuda").manual_seed(2)
    rows = N * T * H * W
    st = ops.BNState.alloc(cin, Cip, 2, rows // 2, "cuda")
    sc = torch.zeros(2, Cip, device="cuda")
    sh = torch.zeros(2, Cip, device="cuda")
    sc[:, :cin] = torch.randn(2, cin, device="cuda", generator=gen)          # negative scales too (glorot'ed gamma)
    sh[:, :cin] = torch.randn(2, cin, device="cuda", generator=gen) * 0.5
    st.scale.copy_(sc.view(-1))
    st.shift.copy_(sh.view(-1))
    act = torch.empty_like(raw)
    ops.bn_apply(raw, st, act, relu=True)
    w = torch.randn(cout, cin, *kernel, device="cuda", generator=gen) / (cin * geom.taps) ** 0.5
    wp = torch.empty(Cop, geom.taps * ops.pad64(Cip), device="cuda", dtype=torch.bfloat16)
    ops.pack_weight(w, wp)
    To, Ho, Wo = geom.out_dims(T, H, W)
    res = {}
    outs, sts, plans = [], [], []
    for x, pro in ((act, None), (raw, st)):
        out = torch.full((N, To, Ho, Wo, Cop), float("nan"), device="cuda", dtype=torch.bfloat16)
        so = ops.BNState.alloc(cout, Cop, 2, N * To * Ho * Wo // 2, "cuda") if with_stats else None
        plan = ops.conv_fwd_plan(x, wp, out, geom, stats=so, prologue=pro)
        plan.run()
        if so is not None:
            res["stat_blocks"] = getattr(plan, "stat_blocks", 0)
            gam, bet = torch.ones(cout, device="cuda"), torch.zeros(cout, device="cuda")
            ops.bn_forward_stats(out, so, gam, bet, None, None, fused_blocks=getattr(plan, "stat_blocks", 0))
        outs.append(out)
        sts.append(so)
        plans.append(plan)
    torch.cuda.synchronize()
    res["kernel"] = ops.kernel_name(plans[1])
    res["fwd_nan"] = int(torch.isnan(outs[1].float()).sum().item())
    res["fwd_equal"] = bool(torch.equal(outs[0], outs[1]))
    res["fwd_rel"] = _rel(outs[1], outs[0])
    if with_stats:
        res["stats_equal"] = bool(torch.equal(sts[0].mean, sts[1].mean) and torch.equal(sts[0].invstd, sts[1].invstd))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for tag, plan in (("fwd_ms_plain", plans[0]), ("fwd_ms_fused", plans[1])):
        for _ in range(2):
            plan.run()
        e0.record()
        for _ in range(iters):
            plan.run()
        e1.record()
        torch.cuda.synchronize()
        res[tag] = e0.elapsed_time(e1) / iters
    e0.record()
    for _ in range(iters):
        ops.bn_apply(raw, st, act, relu=True)
    e1.record()
    torch.cuda.synchronize()
    res["bn_apply_ms"] = e0.elapsed_time(e1) / iters
    # weight gradient
    g = _mk_act(N, To, Ho, Wo, cout, Cop, 3)
    part = torch.empty(64 * 1024 * 1024, device="cuda", dtype=torch.float32)
    dws = []
    for tag, x, pro in (("wgrad_ms_plain", act, None), ("wgrad_ms_fused", raw, st)):
        spec = ops.wgrad_plan(x, g, geom, cout, cin, part, prologue=pro)
        dw = torch.full_like(w, float("nan"))
        spec.run(dw)
        torch.cuda.synchronize()
        dws.append(dw)
        e0.record()
        for _ in range(iters):
            spec.run(dw)
        e1.record()
        torch.cuda.synchronize()
        res[tag] = e0.elapsed_time(e1) / iters
        res["wgrad_kernel"] = ops.kernel_name(spec)
    res["wgrad_nan"] = int(torch.isnan(dws[1]).sum().item())
    res["wgrad_equal"] = bool(torch.equal(dws[0], dws[1]))
    res["wgrad_rel"] = _rel(dws[1], dws[0])
    return res


def case_linear(B, cin, cout):
    import torch
    from cstp_b200 import ops
    Cip, Cop = ops.pad16(cin), ops.pad16(cout)
    gen = torch.Generator(device="cuda").manual_seed(5)
    x = torch.zeros(B, Cip, device="cuda", dtype=torch.bfloat16)
    x[:, :cin] = torch.randn(B, cin, device="cuda", generator=gen).to(torch.bfloat16)
    w = torch.randn(cout, cin, device="cuda", generator=gen) / cin ** 0.5
    b = torch.zeros(Cop, device="cuda")
    b[:cout] = torch.randn(cout, device="cuda", generator=gen)
    wp = torch.empty(Cop, ops.pad64(Cip), device="cuda", dtype=torch.bfloat16)
    ops.pack_weight(w, wp)
    out = torch.full((B, Cop), float("nan"), device="cuda", dtype=torch.bfloat16)
    outf = torch.full((B, Cop), float("nan"), device="cuda", dtype=torch.float32)
    ops.linear_plan(x, wp, out, out_f32=outf, bias=b).run()
    torch.cuda.synchronize()
    ref = x[:, :cin].float() @ w.to(torch.bfloat16).float().t() + b[:cout]
    return {"bf16_rel": _rel(out[:, :cout], ref), "f32_rel": _rel(outf[:, :cout], ref),
            "nan": int(torch.isnan(outf).sum().item())}


def case_elementwise():
    import torch
    import torch.nn.functional as F
    from cstp_b200 import ops
    res = {}
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(7)
    # BN forward/backward vs torch on two groups
    for (rows, C) in [(2 * 3136, 144), (2 * 40, 4096), (2 * 512, 83)]:
        Cp = ops.pad16(C)
        raw = torch.zeros(rows, Cp, device=dev, dtype=torch.bfloat16)
        raw[:, :C] = (torch.randn(rows, C, device=dev, generator=gen) * 1.7 + 0.3).to(torch.bfloat16)
        gamma = torch.randn(C, device=dev, generator=gen)
        beta = torch.randn(C, device=dev, generator=gen)
        rm, rv = torch.zeros(C, device=dev), torch.ones(C, device=dev)
        st = ops.BNState.alloc(C, Cp, 2, rows // 2, dev)
        ops.bn_forward_stats(raw, st, gamma, beta, rm, rv)
        act = torch.empty_like(raw)
        ops.bn_apply(raw, st, act, relu=True)
        xr = raw[:, :C].float().view(2, rows // 2, C).requires_grad_(True)
        rm_ref, rv_ref = torch.zeros(C, device=dev), torch.ones(C, device=dev)
        outs = []
        for gidx in range(2):
            outs.append(F.relu(F.batch_norm(xr[gidx], rm_ref, rv_ref, gamma, beta, True, 0.1, 1e-5)))
        ref = torch.cat(outs, 0)
        tag = f"bn{C}"
        res[tag + "_fwd_rel"] = _rel(act[:, :C], ref)
        res[tag + "_rm_rel"] = _rel(rm, rm_ref)
        res[tag + "_rv_rel"] = _rel(rv, rv_ref)
        d = torch.zeros(rows, Cp, device=dev, dtype=torch.bfloat16)
        d[:, :C] = torch.randn(rows, C, device=dev, generator=gen).to(torch.bfloat16)
        ref.backward(d[:, :C].float())
        dgam, dbet = torch.empty(C, device=dev), torch.empty(C, device=dev)
        gout = torch.empty_like(raw)
        # mask by the *reference* relu output sign is identical to act>0 except at bf16 ties
        ops.bn_backward(d, act, raw, st, gamma, dgam, dbet, gout)
        torch.cuda.synchronize()
        gam_g = torch.autograd.grad(torch.cat([F.relu(F.batch_norm(xr[i], None, None, gamma.requires_grad_(True), beta.requires_grad_(True), True, 0.1, 1e-5)) for i in range(2)], 0), [gamma, beta], d[:, :C].float())
        res[tag + "_dx_rel"] = _rel(gout[:, :C], xr.grad.view(rows, C))
        res[tag + "_dgamma_rel"] = _rel(dgam, gam_g[0])
        res[tag + "_dbeta_rel"] = _rel(dbet, gam_g[1])
    # stem over packed rows (cstp_stem_pack + seven-tap stride-2 implicit GEMM + weight gradient in the stem layout):
    # odd frame height / partial tiles, against conv3d on the bf16-rounded clip
    from cstp_b200.ops import STEM_GEOM, STEM_CHANNELS
    x = torch.rand(3, 3, 2, 22, 36, device=dev, generator=gen) * 2 - 1
    N_, _, T_, H_, W_ = x.shape
    P = torch.full((N_, T_, H_ // 2, W_ // 2, STEM_CHANNELS), 7.0, device=dev, dtype=torch.bfloat16)
    ops.stem_pack(x, P)
    xb = x.to(torch.bfloat16).float()
    taps = F.pad(xb, (3, 3)).unfold(4, 7, 2).permute(0, 2, 3, 4, 5, 1).reshape(N_, T_, H_ // 2, 2, W_ // 2, 21)
    P6 = P.view(N_, T_, H_ // 2, W_ // 2, 2, 32).permute(0, 1, 2, 4, 3, 5)
    res["stem_pack_exact"] = bool(torch.equal(P6[..., :21].float(), taps) and (P6[..., 21:] == 0).all().item())
    w = torch.randn(83, 3, 1, 7, 7, device=dev, generator=gen)
    wb = w.to(torch.bfloat16).float().requires_grad_(True)
    wp = torch.empty(96, 4 * 64, device=dev, dtype=torch.bfloat16)
    ops.pack_weight(w, wp, transpose=2)
    Ho_, Wo_ = H_ // 2, W_ // 2
    raw = torch.empty(N_, T_, Ho_, Wo_, 96, device=dev, dtype=torch.bfloat16)
    ops.conv_fwd_plan(P, wp, raw, STEM_GEOM).run()
    ref = F.conv3d(xb, wb, stride=(1, 2, 2), padding=(0, 3, 3))
    res["stem_fwd_rel"] = _rel(raw[..., :83].float().permute(0, 4, 1, 2, 3), ref)
    res["stem_fwd_padzero"] = bool((raw[..., 83:] == 0).all().item())
    g = torch.zeros_like(raw)
    g[..., :83] = torch.randn(N_, T_, Ho_, Wo_, 83, device=dev, generator=gen).to(torch.bfloat16)
    ref.backward(g[..., :83].float().permute(0, 4, 1, 2, 3))
    scratch = torch.empty(ops.wgrad_partials_need(tuple(P.shape), tuple(g.shape), STEM_GEOM), device=dev)
    dw = torch.full((83, 3, 1, 7, 7), 9.0, device=dev)
    ops.wgrad_plan(P, g, STEM_GEOM, 83, STEM_CHANNELS, scratch, layout=1).run(dw)
    torch.cuda.synchronize()
    res["stem_wgrad_rel"] = _rel(dw, wb.grad)
    # EMA bit-exactness vs torch CPU semantics, SGD vs torch.optim.SGD
    k = torch.randn(1000003, device=dev, generator=gen)
    q = torch.randn(1000003, device=dev, generator=gen)
    kc, qc = k.cpu(), q.cpu()
    kbuf = torch.empty(1000004, device=dev)[:1000003]
    kbuf.copy_(k)
    ops.ema_update(kbuf, q, 0.996)
    refk = kc * 0.996 + qc * (1. - 0.996)
    res["ema_bitexact"] = bool(torch.equal(kbuf.cpu(), refk))
    p = torch.randn(500001, device=dev, generator=gen)
    gr = torch.randn(500001, device=dev, generator=gen) * 0.1
    pr = p.clone().cpu().requires_grad_(True)
    opt = torch.optim.SGD([pr], lr=0.03, momentum=0.9, weight_decay=5e-4)
    mom = torch.zeros_like(p)
    ws = torch.empty(2048, device=dev)
    nout = torch.zeros(2, device=dev)
    pc = p.clone()
    for step in range(2):
        pr.grad = gr.cpu().clone()
        torch.nn.utils.clip_grad_norm_([pr], 18)
        opt.step()
        ops.sgd_clip_step(pc, gr, mom, 0.03, 0.9, 5e-4, 18.0, True, step == 0, nout, ws)
    torch.cuda.synchronize()
    res["sgd_rel"] = _rel(pc.cpu(), pr.detach())
    res["sgd_norm"] = [nout[0].item(), gr.norm().item()]
    return res


def case_losses():
    import torch
    import torch.nn.functional as F
    from cstp_b200 import ops
    dev = "cuda"
    gen = torch.Generator(device=dev).manual_seed(11)
    res = {}
    B, D = 60, 512
    pred = torch.randn(2 * B, D, device=dev, generator=gen).requires_grad_(True)
    tp = torch.randn(2 * B, D, device=dev, generator=gen)
    def lf(x, y):
        return 2 - 2 * (F.normalize(x, dim=-1) * F.normalize(y, dim=-1)).sum(-1)
    ref = (lf(pred[:B], tp[B:]) + lf(pred[B:], tp[:B])).mean()
    up = torch.tensor([0.1], device=dev)
    (ref * 0.1).backward()
    lo = torch.zeros(1, device=dev)
    dp = torch.empty(2 * B, D, device=dev)
    ops.byol_loss(pred.detach(), tp, B, D, lo, up, dp)
    res["byol_loss_rel"] = abs(lo.item() - ref.item()) / abs(ref.item())
    res["byol_grad_rel"] = _rel(dp, pred.grad)
    # CE
    logits = [torch.zeros(B, 16, device=dev) for _ in range(6)]
    for l in logits:
        l[:, :5] = torch.randn(B, 5, device=dev, generator=gen)
    labels = [torch.randint(0, 5 if i < 2 else 4, (B,), device=dev, generator=gen) for i in range(6)]
    w5 = torch.tensor([0.1, 1.0, 0.7, 1.3, 0.9], device=dev)
    lr_ = [l[:, :5].clone().requires_grad_(True) for l in logits]
    ces = [F.cross_entropy(a, b) for a, b in zip(lr_, labels)]
    tot = w5[1] * ces[0] + w5[2] * ces[1] + w5[3] * (ces[2] + ces[3]) + w5[4] * (ces[4] + ces[5])
    tot.backward()
    dl = [torch.empty(B, 16, device=dev) for _ in range(6)]
    lout = torch.zeros(7, device=dev)
    ops.pretext_ce(logits, labels, dl, B, 5, w5, lout)
    res["ce_loss_rel"] = max(abs(lout[i].item() - ces[i].item()) / ces[i].item() for i in range(6))
    res["ce_total_rel"] = abs(lout[6].item() - tot.item()) / tot.item()
    res["ce_grad_rel"] = max(_rel(dl[i][:, :5], lr_[i].grad) for i in range(6))
    # NT-Xent vs closed form in torch fp64
    for rows, d, tau in [(256, 128, 0.1), (1024, 128, 0.1), (200, 96, 0.5)]:
        z = torch.randn(rows, d, device=dev, generator=gen)
        zr = z.double().requires_grad_(True)
        zn = zr / zr.norm(dim=1, keepdim=True).clamp_min(1e-8)
        S = zn @ zn.t() / tau
        N_ = rows // 2
        idx = torch.arange(rows, device=dev)
        pos = (idx + N_) % rows
        Sm = S.masked_fill(torch.eye(rows, device=dev, dtype=torch.bool), float("-inf"))
        lref = (torch.logsumexp(Sm, 1) - S[idx, pos]).mean()
        lref.backward()
        lo = torch.zeros(1, device=dev)
        dz = torch.empty_like(z)
        ws = torch.empty(3 * rows + rows * d, device=dev)          # small workspace: the fp32 SIMT path
        ops.ntxent(z, tau, True, lo, dz, ws)
        torch.cuda.synchronize()
        res[f"ntxent{rows}_loss_rel"] = abs(lo.item() - lref.item()) / lref.item()
        res[f"ntxent{rows}_grad_rel"] = _rel(dz, zr.grad)
    return res


CASES = {
    # name: (fn, kwargs)
    "conv2_spatial_small": ("conv", dict(N=2, T=2, H=56, W=56, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "conv2_temporal_small": ("conv", dict(N=2, T=4, H=56, W=56, cin=144, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "conv3_spatial_s2": ("conv", dict(N=2, T=4, H=56, W=56, cin=64, cout=230, kernel=(1, 3, 3), stride=(1, 2, 2), pad=(0, 1, 1))),
    "conv3_temporal_s2": ("conv", dict(N=2, T=8, H=28, W=28, cin=230, cout=128, kernel=(3, 1, 1), stride=(2, 1, 1), pad=(1, 0, 0))),
    "ds_spatial": ("conv", dict(N=2, T=4, H=56, W=56, cin=64, cout=42, kernel=(1, 1, 1), stride=(1, 2, 2), pad=(0, 0, 0))),
    "ds_temporal": ("conv", dict(N=2, T=8, H=28, W=28, cin=42, cout=128, kernel=(1, 1, 1), stride=(2, 1, 1), pad=(0, 0, 0))),
    "conv5_spatial": ("conv", dict(N=3, T=2, H=7, W=7, cin=512, cout=1152, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "conv5_temporal": ("conv", dict(N=3, T=2, H=7, W=7, cin=1152, cout=512, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "conv4_spatial_s2": ("conv", dict(N=3, T=8, H=28, W=28, cin=128, cout=460, kernel=(1, 3, 3), stride=(1, 2, 2), pad=(0, 1, 1))),
    "stem_temporal": ("conv", dict(N=1, T=8, H=56, W=56, cin=83, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "conv2_spatial_big": ("conv", dict(N=8, T=16, H=56, W=56, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "conv2_temporal_big": ("conv", dict(N=8, T=16, H=56, W=56, cin=144, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "conv3_spatial_big": ("conv", dict(N=8, T=8, H=28, W=28, cin=128, cout=288, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    # enough tiles for conv_gemm's CTA pairs (clusters of two, weight tiles multicast); odd M-tile counts leave the last pair
    # with one CTA beyond the tile space
    "conv4_spatial_pairs": ("conv", dict(N=24, T=4, H=14, W=14, cin=256, cout=576, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "conv5_temporal_pairs": ("conv", dict(N=61, T=2, H=7, W=7, cin=1152, cout=512, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "conv4_spatial_s2_pairs": ("conv", dict(N=15, T=8, H=28, W=28, cin=128, cout=460, kernel=(1, 3, 3), stride=(1, 2, 2), pad=(0, 1, 1))),
    "conv3_temporal_s2_pairs": ("conv", dict(N=21, T=8, H=28, W=28, cin=230, cout=128, kernel=(3, 1, 1), stride=(2, 1, 1), pad=(1, 0, 0))),
    # operand prologue (BatchNorm + ReLU applied to the staged operand): every kernel / layout that carries it
    "pro_conv2_spatial": ("prologue", dict(N=2, T=4, H=56, W=56, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "pro_conv2_temporal": ("prologue", dict(N=2, T=8, H=56, W=56, cin=144, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0), with_stats=True)),
    "pro_stem_temporal": ("prologue", dict(N=2, T=8, H=56, W=56, cin=83, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0), with_stats=True)),
    # 3x1x1 forward with the fused statistics: the network's 16 frames, 32- / 16-channel operand tails, partial tiles along h / w
    "pro_stem_temporal_t16": ("prologue", dict(N=4, T=16, H=56, W=56, cin=83, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0), with_stats=True)),
    "pro_temporal_tail16": ("prologue", dict(N=2, T=4, H=28, W=28, cin=80, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0), with_stats=True)),
    "pro_temporal_ragged": ("prologue", dict(N=4, T=6, H=36, W=28, cin=144, cout=64, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0), with_stats=True)),
    "pro_conv3_temporal_s2": ("prologue", dict(N=2, T=8, H=28, W=28, cin=230, cout=128, kernel=(3, 1, 1), stride=(2, 1, 1), pad=(1, 0, 0))),
    "pro_conv3_spatial": ("prologue", dict(N=2, T=4, H=28, W=28, cin=128, cout=288, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "pro_conv3_temporal": ("prologue", dict(N=2, T=4, H=28, W=28, cin=288, cout=128, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "pro_conv4_spatial": ("prologue", dict(N=4, T=2, H=14, W=14, cin=256, cout=576, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "pro_conv5_spatial": ("prologue", dict(N=6, T=2, H=7, W=7, cin=512, cout=1152, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "pro_conv5_temporal": ("prologue", dict(N=6, T=2, H=7, W=7, cin=1152, cout=512, kernel=(3, 1, 1), stride=(1, 1, 1), pad=(1, 0, 0))),
    "pro_ds_temporal": ("prologue", dict(N=2, T=8, H=28, W=28, cin=42, cout=128, kernel=(1, 1, 1), stride=(2, 1, 1), pad=(0, 0, 0))),
    "pro_ragged": ("prologue", dict(N=2, T=3, H=10, W=6, cin=42, cout=85, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))),
    "linear_proj1": ("linear", dict(B=60, cin=512, cout=4096)),
    "linear_proj2": ("linear", dict(B=60, cin=4096, cout=512)),
    "linear_head": ("linear", dict(B=4, cin=1024, cout=5)),
    "elementwise": ("elementwise", {}),
    "losses": ("losses", {}),
}


def run_case(name):
    kind, kw = CASES[name]
    fn = {"conv": case_conv, "linear": case_linear, "elementwise": case_elementwise, "losses": case_losses,
          "prologue": case_prologue}[kind]
    return fn(**kw)


if __name__ == "__main__":
    if len(sys.argv) >= 3 and sys.argv[1] == "--one":
        out = run_case(sys.argv[2])
        print("RESULT " + json.dumps(out))
        sys.exit(0)
    names = sys.argv[1:] or list(CASES)
    summary = {}
    for n in names:
        t0 = time.time()
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", n], capture_output=True, text=True,
                               timeout=240)
            line = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
            if r.returncode == 0 and line:
                summary[n] = json.loads(line[-1][7:])
            else:
                summary[n] = {"error": (r.stderr or r.stdout)[-1500:], "rc": r.returncode}
        except subprocess.TimeoutExpired:
            summary[n] = {"error": "timeout"}
        print(f"== {n} ({time.time() - t0:.1f}s): {json.dumps(summary[n])}", flush=True)
    bad = [n for n, v in summary.items() if "error" in v]
    print("FAILED CASES:", bad)
