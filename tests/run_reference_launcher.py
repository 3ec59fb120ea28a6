"""Runs the UNMODIFIED reference launcher loop (main_byol.py: main_worker -> train_BYOL, imported from the checkout named by
CSTP_REFERENCE, never copied) on top of the cstp_b200 drop-in modules -- TEST INFRASTRUCTURE.

    python tests/run_reference_launcher.py <out_dir>

What is swapped: `models.model` (the launcher's `from models.model import generate_model`) resolves to
cstp_b200.models.model -- the one-line change INTEGRATION.md describes.  What is stubbed: `decord` / `lmdb` (absent here,
imported at the top of data_process/datasets.py), the dataset class (four seeded synthetic items in the launcher's own
format), and CUDA: the launcher is entered at main_worker with opts.cuda = False (main() itself refuses to run without
a GPU, main_byol.py:158-159) and the engine runs on tests/emulate_ops.py in fp32.  Everything else is the reference's:
argparse options (opts.py), train_BYOL's loop body with its six CrossEntropyLoss terms, --loss_weight sum, zero_grad /
backward / clip_grad_norm_(18) / optim.SGD.step, reduce_mean all-reduce, AverageMeters, CosineAnnealingWarmupRestarts
stepped per epoch, and the TSV Logger.  Writes <out_dir>/result.json with the logged rows and the oracle's losses for the
same two steps.
"""
import json
import os
import sys
import types

import torch

REF = os.environ["CSTP_REFERENCE"]          # the reference checkout (tests/test_reference_integration.py)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = sys.argv[1]
B, T, S, EPOCHS = 4, 4, 32, 2

for m in ("decord", "lmdb"):
    sys.modules.setdefault(m, types.ModuleType(m))
sys.modules["decord"].VideoReader = object
sys.modules["decord"].cpu = lambda *a, **k: None
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

from cstp_b200 import engine  # noqa: E402
from tests import emulate_ops  # noqa: E402
engine.ops, engine.ACT_DTYPE = emulate_ops, torch.float32
import cstp_b200.models.model as our_model  # noqa: E402
import models  # noqa: E402,F401   the reference package (its __init__ is empty); only its `model` submodule is replaced
sys.modules["models.model"] = our_model

sys.argv = ["main_byol.py", "--task", "loss_com", "--loss_weight", "0.1", "1", "1", "1", "1", "--model_name", "r21d_byol",
            "--model_depth", "1", "--dataset", "FakeClips", "--batch_size", str(B), "--n_epochs", str(EPOCHS), "--n_workers", "0",
            "--result_path", OUT, "--learning_rate", "0.03", "--weight_decay", "5e-4", "--sample_duration", str(T),
            "--sample_size", str(S)]
import main_byol  # noqa: E402   the reference launcher, unmodified
from opts import parse_opts  # noqa: E402
from oracle import cstp_oracle as O  # noqa: E402

x1, x2, labels = O.structured_batch(B, 0, T, S)


class FakeClips(torch.utils.data.Dataset):
    """Items in the format of UcfRepreBYOLSpPre.__getitem__ (data_process/datasets.py:850-948):
    ((clip_1, clip_2), (spa_label, tem_label, pb_label, (rot_label_1, rot_label_2)))."""

    def __init__(self, data_type, opts, split, sp_transform):
        assert data_type == "train" and sp_transform is not None

    def __len__(self):
        return B

    def __getitem__(self, i):
        spa, tem, pb, r1, r2 = (int(l[i]) for l in labels)
        return (x1[i], x2[i]), (spa, tem, pb, (r1, r2))


main_byol.FakeClips = FakeClips
opts = parse_opts()
assert opts.task == "loss_com" and opts.loss_weight == [0.1, 1.0, 1.0, 1.0, 1.0], opts.loss_weight
# the launcher's own distributed branch with one rank (its non-distributed branch cannot run: get_dataloader returns one
# value there and main_byol.py:207 unpacks two); gloo instead of nccl because this process has no GPU
opts.cuda, opts.distributed, opts.nprocs, opts.world_size, opts.local_rank = False, True, 1, 1, 0
opts.dist_backend, opts.dist_url = "gloo", f"file://{OUT}/rdzv"
torch.manual_seed(opts.manual_seed)

built = {}
_generate = our_model.generate_model


def spy(o):
    r = _generate(o)
    built["model"] = r[0]
    return r


main_byol.generate_model = spy
from cstp_b200.models.pace.r21d_byol import R21DBYOL  # noqa: E402
torch.manual_seed(1)
state = {k: v.clone() for k, v in R21DBYOL(pretrain=True).state_dict().items() if not k.endswith("num_batches_tracked")}
torch.manual_seed(1)                                     # generate_model draws the same initial weights
main_byol.main_worker(0, 1, opts)

log = os.path.join(OUT, "FakeClips", "loss_com", f"FakeClips_train_clip{T}modelr21d_byol1.log")
rows = [l.rstrip("\n").split("\t") for l in open(log)]
# the same two optimiser steps through the oracle (the batch holds every item, so the loader's shuffle only permutes it)
from cstp_b200.engine import trainable_param_specs  # noqa: E402
from cstp_b200.train import epoch_lr  # noqa: E402
trainable = [n for n, _ in trainable_param_specs()]
mom: dict = {}
ref = []
for ep in range(1, EPOCHS + 1):
    r = O.pretrain_step(state, trainable, x1, x2, labels, [0.1, 1, 1, 1, 1], epoch_lr(ep, EPOCHS, 0.03), mom)
    ref.append({"loss": r["loss_total"], "loss_byol": r["loss_byol"], "ce": r["ce"]})
m = built["model"]
inner = getattr(m, "module", m)
w = "online_net.conv3.block1.conv1.spatial_conv.weight"
json.dump({"rows": rows, "oracle": ref, "wrapper": type(m).__name__,
           "model_class": type(inner).__module__ + "." + type(inner).__name__,
           "weight_rel": ((dict(inner.named_parameters())[w].detach() - state[w]).norm() / state[w].norm()).item()},
          open(os.path.join(OUT, "result.json"), "w"))
torch.distributed.destroy_process_group()
