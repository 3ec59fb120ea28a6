"""Step time of the pretraining step with its forward / backward / update split (CUDA events on the main stream).
Development tool for schedule experiments; the engine options of the DESIGN.md appendix come from the environment
(CSTP_FUSE_POLICY, CSTP_FUSE_MIN_POSITIONS, ...) and are echoed in the result line.
    python tools/step_time.py [B] [--no-overlap] [--no-graph] [--steps K]"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from cstp_b200.models.pace.r21d_byol import R21DBYOL  # noqa: E402
from cstp_b200.synthetic import synthetic_batch  # noqa: E402

args = [a for a in sys.argv[1:] if not a.startswith("--")]
B = int(args[0]) if args else 60
K = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 8
torch.manual_seed(1)
m = R21DBYOL(pretrain=True).cuda()
m.engine_options = {}
if "--no-overlap" in sys.argv:
    m.engine_options["overlap"] = False
if "--no-graph" in sys.argv:
    m.engine_options["graph"] = False
x1, x2, labels = synthetic_batch(B, 0)
x1, x2 = x1.cuda(), x2.cuda()
labels = tuple(l.cuda() for l in labels)
lw = (0.1, 1, 1, 1, 1)
for _ in range(3):
    m.train_step(x1, x2, labels, lw, lr=0.03)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(K):
    out = m.train_step(x1, x2, labels, lw, lr=0.03)
b.record()
torch.cuda.synchronize()
whole = a.elapsed_time(b) / K
eng = m._engine
ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
for k in range(K):
    ev[k][0].record()
    eng.forward(x1, x2)
    eng.pretext_losses(labels)
    ev[k][1].record()
    eng.backward()
    ev[k][2].record()
    eng.optimizer_step(0.03, 0.9, 5e-4, 18.0, True)
    ev[k][3].record()
torch.cuda.synchronize()
seg = [sum(ev[k][i].elapsed_time(ev[k][i + 1]) for k in range(K)) / K for i in range(3)]
print(json.dumps({"B": B, "ms_per_step": round(whole, 3), "fwd": round(seg[0], 3), "bwd": round(seg[1], 3),
                  "update": round(seg[2], 3), "losses": [round(v, 5) for v in out.tolist()],
                  "env": {k: v for k, v in os.environ.items() if k.startswith("CSTP_")}}), flush=True)
