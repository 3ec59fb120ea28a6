"""The reference's own launcher and checkpoints against the drop-in modules (SURVEY.md 8 f-3 / f-4, a15).

Two tests execute the UNMODIFIED reference (a checkout of KT27-A/CSTP named by the CSTP_REFERENCE environment variable,
imported in a subprocess, never copied) and skip where no such checkout is given.  The checkpoint hand-off is also checked
without it, against the state_dict keys, parameter order and shapes the reference recorded in tests/golden/step_b2.pt
(oracle/make_golden.py) and the CPU oracle that tests/test_oracle_golden.py pins to the reference's own outputs.  The
CUDA path is covered by tests/test_gpu_*.py.
The engine runs on tests/emulate_ops.py in fp32: what is under test is the integration surface (generate_model, the DDP
wrap, autograd through the drop-in forward, optim.SGD on the aliased parameters, checkpoint formats), which is host code.
"""
import json
import os
import subprocess
import sys
import types

import pytest
import torch

REF = os.environ.get("CSTP_REFERENCE", "")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
needs_reference = pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "main_byol.py")),
                                     reason="needs a checkout of the reference KT27-A/CSTP named by CSTP_REFERENCE")
LW = (0.1, 1.0, 1.0, 1.0, 1.0)


def _run(script, out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", script), str(out)], capture_output=True, text=True,
                       timeout=1500, cwd=ROOT)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    return json.load(open(os.path.join(out, "result.json")))


@needs_reference
def test_unmodified_launcher_trains_on_the_dropin_backend(tmp_path):
    """main_byol.py (main_worker + train_BYOL, argparse options, DistributedSampler loader, DDP-wrapped model from
    generate_model, CrossEntropyLoss x 6, --loss_weight, clip_grad_norm_, optim.SGD, cosine schedule, TSV Logger) for two
    epochs: every logged column equals the oracle's value for the same two optimiser steps."""
    res = _run("run_reference_launcher.py", tmp_path)
    assert res["wrapper"] == "DistributedDataParallel"                 # generate_model's DDP wrap (models/model.py:97-103)
    assert res["model_class"] == "cstp_b200.models.pace.r21d_byol.R21DBYOL"
    rows = res["rows"]
    assert rows[0] == ["epoch", "loss", "loss_byol", "loss_pred_spa", "loss_pred_tem", "loss_pred_pb", "loss_pred_rot", "acc", "lr"]
    assert [r[0] for r in rows[1:]] == ["1", "2"]
    assert rows[1][8] == "1e-05" and rows[2][8] == "0.03"              # epoch 1 runs at min_lr (main_byol.py:252-258)
    for row, ref in zip(rows[1:], res["oracle"]):
        got = [float(v) for v in row[1:7]]
        want = [ref["loss"], ref["loss_byol"], ref["ce"][0], ref["ce"][1], (ref["ce"][2] + ref["ce"][3]) / 2,
                (ref["ce"][4] + ref["ce"][5]) / 2]                         # main_byol.py:81-84: pb / rot columns are means
        assert all(abs(a - b) < 1e-5 * abs(b) for a, b in zip(got, want)), (got, want)
        assert row[7] == ""                                             # "acc": None
    assert res["weight_rel"] < 1e-3                                     # the weights after two SGD steps follow the oracle's


@needs_reference
def test_checkpoints_written_by_the_reference_and_by_us_are_interchangeable(tmp_path):
    res = _run("run_reference_checkpoint.py", tmp_path)
    assert res["resume_epoch"] == 100                                   # main_byol.py:214-215: parsed from the file name
    assert res["weights_equal_after_load"] and res["momentum_equal_after_load"]
    for a, b in ((res["ours_step2"], res["ref_step2"]), (res["ours_step3"], res["ref2_step3"])):
        assert abs(a[0] - b[0]) < 1e-5 * b[0] and abs(a[1] - b[1]) < 1e-5 * b[1], (a, b)
    assert res["weights_rel_after_step2"] < 2e-2 and res["weights_rel_after_step3"] < 2e-2
    missing, unexpected, epoch, arch = res["ref_loads_ours"]
    assert missing == [] and unexpected == [] and epoch == 102 and arch == "r21d_byol-1"
    assert res["ft_backbone_equal"]                                     # neq_load_customized: online_net.* carried over
    assert res["ft_head_keys"] == ["classify.bias", "classify.weight", "cls_bn.bias", "cls_bn.num_batches_tracked",
                                   "cls_bn.running_mean", "cls_bn.running_var", "cls_bn.weight"]


def _reference_layout_checkpoint(path, g, state, mom):
    """A checkpoint as main_byol.py:132-140 writes it for the reference model: `module.` keys in the order of the
    reference's state_dict and optim.SGD(model.parameters()).state_dict() over the reference's parameter order (both
    recorded from the reference in tests/golden/step_b2.pt), with momentum buffers for the parameters in `mom`."""
    params = [torch.nn.Parameter(state[n].clone()) for n in g["param_names"]]
    opt = torch.optim.SGD(params, lr=0.03, momentum=0.9, weight_decay=5e-4)          # main_byol.py:229-232
    for p, n in zip(params, g["param_names"]):
        if n in mom:
            opt.state[p]["momentum_buffer"] = mom[n].clone()
    sd = {"module." + k: state[k].clone() for k in g["state_dict_keys"]}
    torch.save({"epoch": 101, "arch": "r21d_byol-1", "state_dict": sd, "optimizer": opt.state_dict()}, path)


def test_checkpoints_interchange_in_the_reference_layout(emulated_engine, tmp_path, monkeypatch):
    """Without a reference checkout: resume from a checkpoint in the reference's layout (weights, BatchNorm buffers and
    the momentum of EVERY trainable parameter land where the reference's SGD kept them), take the step the oracle takes
    from the same state, write our checkpoint and load it the way the reference does (strict key set, shapes,
    optimizer.load_state_dict over the reference's parameter order), and hand it to the finetune model."""
    from cstp_b200 import train as TR
    from cstp_b200.engine import trainable_param_specs
    from cstp_b200.models.model import generate_model
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    from oracle import cstp_oracle as O
    from tests.parity import load_golden, rel
    monkeypatch.setattr(emulated_engine, "ACT_DTYPE", torch.float32)
    g = load_golden("step_b2.pt")
    B, T, S = 4, 4, 32
    x1, x2, labels = O.structured_batch(B, 0, T, S)
    torch.manual_seed(1)
    state = {k: v.clone() for k, v in R21DBYOL(pretrain=True).state_dict().items()}
    trainable = [n for n, _ in trainable_param_specs()]
    gen = torch.Generator().manual_seed(5)
    mom = {n: 0.01 * torch.randn(state[n].shape, generator=gen) for n in trainable}
    path = str(tmp_path / "save_100.pth")
    _reference_layout_checkpoint(path, g, state, mom)

    # ---- resume from the reference's layout
    o = types.SimpleNamespace(model_name="r21d_byol", task="resume", distributed=False, device="cpu", arch="r21d_byol-1",
                              resume_md_path=path, n_classes=101)
    ours, _ = generate_model(o)
    ours.train()
    assert TR.load_checkpoint(path, ours, example_clip=x1) == 100                    # main_byol.py:214-215
    assert all(torch.equal(v, state[k]) for k, v in ours.state_dict().items())
    eng = ours._engine
    assert not eng.first_step
    assert all(torch.equal(eng.train.view(n, eng.mom), mom[n]) for n in trainable)

    # ---- the next step uses that momentum: the oracle's step from the same weights and momentum buffers
    l = ours.train_step(x1, x2, labels, LW, lr=0.03, momentum=0.9, weight_decay=5e-4, clip_grad_norm=18.0)
    ref_state = {k: v.clone() for k, v in state.items() if not k.endswith("num_batches_tracked")}
    ref_mom = {n: v.clone() for n, v in mom.items()}
    ref = O.pretrain_step(ref_state, trainable, x1, x2, labels, list(LW), 0.03, ref_mom)
    assert abs(LW[0] * l[7].item() + l[6].item() - ref["loss_total"]) < 1e-5 * ref["loss_total"]
    assert abs(l[7].item() - ref["loss_byol"]) < 1e-5 * ref["loss_byol"]
    sd = ours.state_dict()
    worst = max(rel(sd[k], v) for k, v in ref_state.items())
    assert worst < 1e-2, worst                                  # 2.4e-3 measured; ~10 if the momentum were dropped

    # ---- our checkpoint, loaded the way the reference loads it (models/model.py:116-120, main_byol.py:243-244)
    path2 = str(tmp_path / "save_101.pth")
    TR.save_checkpoint(path2, ours, 101, "r21d_byol-1", lr=0.03, momentum=0.9, weight_decay=5e-4)
    ck = torch.load(path2, weights_only=False)
    assert (ck["epoch"], ck["arch"]) == (102, "r21d_byol-1")
    assert list(ck["state_dict"]) == ["module." + k for k in g["state_dict_keys"]]    # strict load: no missing / unexpected
    assert all(tuple(ck["state_dict"]["module." + n].shape) == tuple(s) for n, s in g["param_shapes"].items())
    params = [torch.nn.Parameter(torch.zeros(g["param_shapes"][n])) for n in g["param_names"]]
    opt = torch.optim.SGD(params, lr=0.03, momentum=0.9, weight_decay=5e-4)
    opt.load_state_dict(ck["optimizer"])
    for p, n in zip(params, g["param_names"]):
        if n.startswith("target_net."):
            assert p not in opt.state, n                                               # the EMA target is not optimised
        else:
            assert torch.equal(opt.state[p]["momentum_buffer"], eng.train.view(n, eng.mom)), n

    # ---- pretrain -> finetune hand-off from the reference's layout (neq_load_customized)
    o = types.SimpleNamespace(model_name="r21d_byol", task="ft_all", distributed=False, device="cpu", arch="r21d_byol-1",
                              pretrained_path=path, n_classes=101)
    ft, _ = generate_model(o)
    sd_ft = ft.state_dict()
    assert all(torch.equal(v, state[k]) for k, v in sd_ft.items() if k.startswith("online_net."))
    assert sorted(k for k in sd_ft if not k.startswith("online_net.")) == [
        "classify.bias", "classify.weight", "cls_bn.bias", "cls_bn.num_batches_tracked", "cls_bn.running_mean",
        "cls_bn.running_var", "cls_bn.weight"]
