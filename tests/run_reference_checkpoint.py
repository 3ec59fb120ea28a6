"""Checkpoint hand-off with the UNMODIFIED reference (the checkout named by CSTP_REFERENCE) in both directions -- TEST
INFRASTRUCTURE.

    python tests/run_reference_checkpoint.py <out_dir>

  1. the reference trains one step (models/pace/r21d_byol.py R21DBYOL wrapped the way main_byol.py saves it: `module.`
     keys; optim.SGD) and writes save_100.pth exactly as main_byol.py:132-140 does;
  2. cstp_b200 resumes from that file through generate_model(task='resume') + train.load_checkpoint (weights, BatchNorm
     buffers, SGD momentum) and takes the next step; the reference takes the same step: losses and weights must agree;
  3. cstp_b200 writes save_101.pth (train.save_checkpoint); the reference loads it with its own strict
     load_state_dict + optimizer.load_state_dict (main_byol.py:243-244, models/model.py:116-120) and both take a third step;
  4. pretrain -> finetune hand-off: generate_model(task='ft_all', pretrained_path=save_101.pth) (neq_load_customized).
The engine runs on tests/emulate_ops.py in fp32 (no GPU here).  Writes <out_dir>/result.json.
"""
import json
import os
import sys
import types

import torch

REF = os.environ["CSTP_REFERENCE"]          # the reference checkout (tests/test_reference_integration.py)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = sys.argv[1]
B, T, S = 4, 4, 32
LW = [0.1, 1.0, 1.0, 1.0, 1.0]
sys.path.insert(0, ROOT)

from cstp_b200 import engine  # noqa: E402
from tests import emulate_ops  # noqa: E402
engine.ops, engine.ACT_DTYPE = emulate_ops, torch.float32
from cstp_b200 import train as TR  # noqa: E402
from cstp_b200.models.model import generate_model  # noqa: E402
from oracle import cstp_oracle as O  # noqa: E402

sys.path.insert(1, REF)
from models.pace import r21d_byol as ref_mod  # noqa: E402   the reference, unmodified

x1, x2, labels = O.structured_batch(B, 0, T, S)
crit = torch.nn.CrossEntropyLoss()


def ref_step(model, opt):
    """main_byol.py:60-91."""
    loss_byol, p = model(x1, x2, o_type="loss_com")
    loss_byol = loss_byol.mean()
    spa, tem, pb, r1, r2 = labels
    total = (LW[0] * loss_byol + LW[1] * crit(p[0], spa) + LW[2] * crit(p[1], tem) + LW[3] * crit(p[2], pb) + LW[3] * crit(p[3], pb)
             + LW[4] * crit(p[4], r1) + LW[4] * crit(p[5], r2))
    opt.zero_grad()
    total.backward()
    torch.nn.utils.clip_grad_norm_(model.parameters(), 18)
    opt.step()
    return total.item(), loss_byol.item()


def our_step(model):
    l = model.train_step(x1, x2, labels, LW, lr=0.03, momentum=0.9, weight_decay=5e-4, clip_grad_norm=18.0)
    return LW[0] * l[7].item() + l[6].item(), l[7].item()


def rel(a, b):
    return ((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-30)).item()


res = {}
# ---- 1. the reference writes a checkpoint
torch.manual_seed(1)
ref = torch.nn.DataParallel(ref_mod.R21DBYOL(pretrain=True))         # the wrapper only contributes the `module.` key prefix
ref.train()
opt = torch.optim.SGD(ref.parameters(), lr=0.03, momentum=0.9, weight_decay=5e-4)        # main_byol.py:229-232
res["ref_step1"] = ref_step(ref, opt)
path = os.path.join(OUT, "save_100.pth")
torch.save({"epoch": 101, "arch": "r21d_byol-1", "state_dict": ref.state_dict(), "optimizer": opt.state_dict()}, path)
# ---- 2. cstp_b200 resumes from it
o = types.SimpleNamespace(model_name="r21d_byol", task="resume", distributed=False, device="cpu", arch="r21d_byol-1",
                          resume_md_path=path, n_classes=101)
ours, _ = generate_model(o)
ours.train()
res["resume_epoch"] = TR.load_checkpoint(path, ours, example_clip=x1)
sd_ref = {k[len("module."):]: v for k, v in ref.state_dict().items()}
res["weights_equal_after_load"] = all(torch.equal(v, sd_ref[k]) for k, v in ours.state_dict().items())
names = [n for n, _ in ours.named_parameters()]
i = names.index("online_net.conv4.block1.conv2.temporal_conv.weight")
res["momentum_equal_after_load"] = bool(torch.equal(ours._engine.train.view(names[i], ours._engine.mom),
                                                    opt.state[list(ref.parameters())[i]]["momentum_buffer"]))
res["ours_step2"] = our_step(ours)
res["ref_step2"] = ref_step(ref, opt)
sd_ref = {k[len("module."):]: v for k, v in ref.state_dict().items()}
res["weights_rel_after_step2"] = max(rel(v, sd_ref[k]) for k, v in ours.state_dict().items() if v.dtype.is_floating_point)
# ---- 3. the reference resumes from OUR checkpoint
path2 = os.path.join(OUT, "save_101.pth")
TR.save_checkpoint(path2, ours, 101, "r21d_byol-1", lr=0.03, momentum=0.9, weight_decay=5e-4)
ck = torch.load(path2, weights_only=False)
torch.manual_seed(7)
ref2 = torch.nn.DataParallel(ref_mod.R21DBYOL(pretrain=True))
ref2.train()
opt2 = torch.optim.SGD(ref2.parameters(), lr=0.03, momentum=0.9, weight_decay=5e-4)
missing = ref2.load_state_dict(ck["state_dict"])                   # strict (models/model.py:119)
opt2.load_state_dict(ck["optimizer"])                              # main_byol.py:243-244
res["ref_loads_ours"] = (list(missing.missing_keys), list(missing.unexpected_keys), ck["epoch"], ck["arch"])
res["ref2_step3"] = ref_step(ref2, opt2)
res["ours_step3"] = our_step(ours)
sd_ref2 = {k[len("module."):]: v for k, v in ref2.state_dict().items()}
res["weights_rel_after_step3"] = max(rel(v, sd_ref2[k]) for k, v in ours.state_dict().items() if v.dtype.is_floating_point)
# ---- 4. pretrain -> finetune hand-off from a reference-format checkpoint
o = types.SimpleNamespace(model_name="r21d_byol", task="ft_all", distributed=False, device="cpu", arch="r21d_byol-1",
                          pretrained_path=path, n_classes=101)
ft, params = generate_model(o)
sd_ft, sd_pre = ft.state_dict(), torch.load(path, weights_only=False)["state_dict"]
res["ft_backbone_equal"] = all(torch.equal(v, sd_pre["module." + k]) for k, v in sd_ft.items() if k.startswith("online_net."))
res["ft_head_keys"] = sorted(k for k in sd_ft if not k.startswith("online_net."))
json.dump(res, open(os.path.join(OUT, "result.json"), "w"), indent=1)
