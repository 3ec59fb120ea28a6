"""`generate_model(opts)` (models/model.py:39-144, r21d_byol branch) on the engine over tests/emulate_ops.py: every task the
factory serves, with and without the DDP wrap (world_size-2 gloo), and DDP-hook gradients against the fused GradSync path."""
import os
import tempfile
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

LW = (0.1, 1.0, 1.0, 1.0, 1.0)
B, T, S = 4, 4, 32


def _opts(**kw):
    base = dict(model_name="r21d_byol", task="loss_com", distributed=False, device="cpu", arch="r21d_byol-1", n_classes=101,
                local_rank=0)
    base.update(kw)
    return types.SimpleNamespace(**base)


def test_tasks_and_errors(emulated_engine, tmp_path):
    from cstp_b200 import train as TR
    from cstp_b200.models.model import generate_model
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from oracle import cstp_oracle as O
    with pytest.raises(ValueError, match="Please check the input backbone!"):      # models/model.py:79
        generate_model(_opts(model_name="resnext"))
    torch.manual_seed(1)
    m, params = generate_model(_opts(task="loss_com"))
    assert isinstance(m, R21DBYOL) and m.pretrain and len(list(params)) == len(list(m.parameters()))
    x1, x2, lab = O.structured_batch(2, 0, T, S)
    m.train_step(x1, x2, lab, LW, lr=0.03)
    ck = str(tmp_path / "save_3.pth")
    TR.save_checkpoint(ck, m, 3, "r21d_byol-1")
    # resume: weights and buffers come back (`module.` prefix stripped for the unwrapped model)
    r, _ = generate_model(_opts(task="resume", resume_md_path=ck))
    sa, sb = m.state_dict(), r.state_dict()
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    with pytest.raises(AssertionError):                                            # models/model.py:119: arch must match
        generate_model(_opts(task="resume", resume_md_path=ck, arch="r21d_byol-2"))
    # ft_all / ft_fc: the backbone is carried over, the head is fresh; ft_fc freezes everything but `classify`
    fa, pa = generate_model(_opts(task="ft_all", pretrained_path=ck))
    assert not fa.pretrain and all(torch.equal(v, sa[k]) for k, v in fa.state_dict().items() if k.startswith("online_net."))
    assert len(list(pa)) == len(list(fa.parameters())) and all(p.requires_grad for p in fa.parameters())
    ff, pf = generate_model(_opts(task="ft_fc", pretrained_path=ck))
    assert [g.get("lr", None) for g in pf].count(0.0) == len(pf) - 2
    assert sorted(n for n, p in ff.named_parameters() if p.requires_grad) == ["classify.bias", "classify.weight"]
    # test: returns the bare model with the finetuned weights loaded
    ft_ck = str(tmp_path / "ft.pth")
    torch.save({"arch": "r21d_byol-1", "state_dict": {"module." + k: v for k, v in fa.state_dict().items()}}, ft_ck)
    t = generate_model(_opts(task="test", test_md_path=ft_ck))
    assert not isinstance(t, tuple) and all(torch.equal(v, fa.state_dict()[k]) for k, v in t.state_dict().items())


def _worker(rank, world, path, out):
    """Two ranks: (a) the reference's loop body on the DDP-wrapped model generate_model returns; (b) the fused train_step
    with GradSync.  Same shards, same seeds."""
    from cstp_b200 import engine, parallel as P
    from cstp_b200.models.model import generate_model
    from oracle import cstp_oracle as O
    from tests import emulate_ops
    engine.ops, engine.ACT_DTYPE = emulate_ops, torch.float32
    torch.set_num_threads(2)
    dist.init_process_group("gloo", init_method=f"file://{path}", rank=rank, world_size=world)
    x1, x2, lab = O.structured_batch(B, 0, T, S)
    lo, hi = P.shard_bounds(B, rank, world)
    x1, x2, lab = x1[lo:hi].contiguous(), x2[lo:hi].contiguous(), tuple(l[lo:hi].contiguous() for l in lab)
    torch.manual_seed(1)
    ddp, params = generate_model(_opts(task="loss_com", distributed=True, local_rank=rank))
    assert type(ddp).__name__ == "DistributedDataParallel"
    opt = torch.optim.SGD(params, lr=0.03, momentum=0.9, weight_decay=5e-4)
    crit = torch.nn.CrossEntropyLoss()
    ddp.train()
    loss_byol, p = ddp(x1, x2, o_type="loss_com")
    spa, tem, pb, r1, r2 = lab
    total = (LW[0] * loss_byol.mean() + crit(p[0], spa) + crit(p[1], tem) + crit(p[2], pb) + crit(p[3], pb) + crit(p[4], r1)
             + crit(p[5], r2))
    opt.zero_grad()
    total.backward()                                     # DDP's reducer averages the gradients of the aliased parameters
    torch.nn.utils.clip_grad_norm_(ddp.parameters(), 18)
    opt.step()
    torch.manual_seed(1)
    fused, _ = generate_model(_opts(task="loss_com"))
    fused.train_step(x1, x2, lab, LW, lr=0.03, grad_sync=P.GradSync())
    torch.save({"ddp": {k: v.clone() for k, v in ddp.module.state_dict().items()},
                "fused": {k: v.clone() for k, v in fused.state_dict().items()}, "loss": total.item()}, f"{out}.{rank}")
    dist.destroy_process_group()


def test_ddp_wrapped_dropin_equals_fused_gradsync_world2(monkeypatch):
    # the ranks run the host logic over the CPU stand-in of the kernel layer: they must see no GPU, or generate_model places
    # rank r on cuda:r (which a one-GPU machine does not have)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    d = tempfile.mkdtemp()
    mp.spawn(_worker, args=(2, os.path.join(d, "rdzv"), os.path.join(d, "out")), nprocs=2, join=True)
    r0, r1 = (torch.load(os.path.join(d, f"out.{r}"), weights_only=False) for r in range(2))
    for k, v in r0["ddp"].items():
        if v.dtype.is_floating_point and "running" not in k:
            assert torch.equal(v, r1["ddp"][k]), k                     # replicas hold identical weights after the DDP step
            ref = r0["fused"][k]
            assert (v - ref).norm() <= 1e-5 * ref.norm().clamp_min(1e-12), k        # and they equal the fused + GradSync step
