"""Static-shape step engine of the B200-native `r21d_byol` pretraining hot path.

The engine owns every device buffer of one pretraining step for a fixed per-GPU batch `B` and clip size
(T, H, W) and turns the reference step (main_byol.py:60-91 around R21DBYOL.forward(o_type="loss_com"),
models/pace/r21d_byol.py:357-382) into three launch programs of hand-written sm_100a kernels:

  forward   online_net(view1|view2) -> predictor -> EMA -> target_net(view1|view2) -> BYOL loss -> pretext heads
  backward  heads / predictor / projector / backbone (BN-bwd, wgrad, dgrad per layer) into ONE flat fp32 grad buffer
  update    (grad all-reduce) -> global-norm clip + SGD momentum (or Adam / AdamW) on the flat buffers -> bf16 weight re-pack

Data layout in HBM
  * parameters: two flat fp32 buffers (trainable = online_net + predictor + 4 pretext heads; target_net), every
    tensor in a 16-float aligned slot; gradients and SGD momentum mirror the trainable buffer (and so do Adam's exp_avg /
    exp_avg_sq, allocated when Adam first runs).  The nn.Parameters of
    the drop-in module are views into these buffers (reference shapes, state_dict compatible).
  * activations: bf16 NDHWC, channels padded to 16, the two views concatenated along N (2B samples) and kept as two
    BatchNorm statistics groups (the reference runs the views one after the other, SURVEY.md 0.3).
  * weights for the tensor cores: bf16 K-major packed copies (forward and transposed-for-dgrad), refreshed after
    every optimiser step / EMA update.

Everything is launched on the current CUDA stream through the C ABI (cstp_b200.ops); torch is only used for
memory, streams and torch.distributed.  There is no CPU path.

Classes: ProgramEngine holds what every engine shares (stores, program builders, backward, weight packs, CUDA-graph
capture); OptimizerEngine adds the fused optimiser; StepEngine is the pretraining step.  The finetune, inference and
backbone engines (engine_ft, engine_backbone) build on the same two bases.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import torch

from . import ops
from .ops import REPR_STATS, ConvGeom, pad16, pad64

import os

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
# conv -> BatchNorm -> ReLU -> conv edges (r21d_byol.py:94-97): the consumer's forward and weight-gradient kernels read the
# producer's RAW output and apply the BatchNorm affine map + ReLU to their staged operand tiles (ops.conv_fwd_plan /
# ops.wgrad_plan `prologue`), so the normalised activation is neither written nor re-read.  "0" restores the standalone
# cstp_bn_apply pass on every edge (same bits either way: tests/test_gpu_step.py).
FUSE_BN_APPLY = os.environ.get("CSTP_FUSE_BN_APPLY", "1") == "1"
# ... for activations with at least this many positions per (sample, frame) plane: the 56 x 56 planes of the stem and
# conv2, where the tensors are 0.8-1.7 GB per network at batch 60 and every edge nets -0.3 to -0.4 ms per step (forward
# of both networks + weight gradient against the two cstp_bn_apply passes saved; profiles/README.md).  On the 28 x 28 planes
# of conv3 the pass saved is worth 0.07-0.15 ms and the consumers lose more than that (shallow TMA pipelines with
# non-resident weights cannot hide the extra hop); on 14 x 14 / 7 x 7 planes the tensors are L2-sized and the 1x3x3
# convolutions re-stage -- and would re-transform -- the same box once per filter tap (csrc/conv_gemm.cu).
FUSE_MIN_POSITIONS = int(os.environ.get("CSTP_FUSE_MIN_POSITIONS") or 56 * 56)
# Which edges: "all": every conv -> BatchNorm -> ReLU -> conv edge above the size threshold; "auto" (default): networks
# without a backward pass defer every such edge, the online network only those in front of a 3x1x1 convolution; "none".
# Background (measured per layer at batch 60, profiles/README.md): the in-place transform costs the consumer's forward
# +1..10 % (1x3x3: nine taps per staged box) to +25 % (3x1x1) and its weight-gradient kernel +35 % (3x1x1, where the
# transformed operand is the N side of the flipped product) to +45 % (1x3x3, where both M classes transform the same box),
# against the two HBM passes of cstp_bn_apply the edge drops: 0.56 ms for a 144-channel 56 x 56 tensor (the input of a
# 3x1x1 layer), 0.25 ms for a 64-channel one (the input of a 1x3x3 layer) -- the latter is less than its weight-gradient
# kernel loses, so edges in front of a 1x3x3 convolution stay materialised where there is a backward pass.
FUSE_POLICY = os.environ.get("CSTP_FUSE_POLICY") or "auto"
# The whole step (forward, losses, backward, gradient all-reduce, optimiser, re-pack: ~560 launches on three streams) is
# captured into ONE CUDA graph after an eager first step and replayed from then on (StepEngine.graphed_step): at 16 samples
# per GPU the eager step is bound by the host issuing launches through ctypes, not by the GPU.  "0": always eager.
USE_GRAPH = os.environ.get("CSTP_GRAPH", "1") == "1"
# Storage type of activations, activation gradients and packed weights.  The CUDA kernels only implement bf16; the
# CPU emulator in tests/ also runs the orchestration in fp32 to separate wiring errors from rounding.
ACT_DTYPE = torch.bfloat16


OPTIMIZERS = ("sgd", "adam", "adamw")


def adam_scalars(step: int, lr, betas, eps, weight_decay, decoupled: bool, max_norm=0.0, clip=False) -> tuple:
    """The cstp_adam_hyper scalars (include/cstp_b200.h, in field order) of Adam / AdamW step `step` (1-based), computed in
    double as torch.optim.Adam(W) computes them (_single_tensor_adam); the kernel receives them rounded to fp32."""
    b1, b2, lr, wd = float(betas[0]), float(betas[1]), float(lr), float(weight_decay)
    return (lr / (1 - b1 ** step), (1 - b2 ** step) ** 0.5, 1 - b1, b2, 1 - b2, float(eps), 0.0 if decoupled else wd,
            1 - lr * wd if decoupled else 1.0, float(max_norm), 1.0 if clip else 0.0)


def intermed_channels(cin: int, cout: int, k: tuple[int, int, int]) -> int:
    """Channel count between the spatial and temporal halves -- models/pace/r21d_byol.py:74-76."""
    kt, kh, kw = k
    return int(math.floor((kt * kh * kw * cin * cout) / (kh * kw * cin + kt * cout)))


# ---------------------------------------------------------------------------------------------- flat parameter store
class FlatStore:
    """name -> fp32 view registry over one flat buffer; every tensor sits in a 16-float aligned, zero-padded slot."""

    def __init__(self, specs, device, dtype=torch.float32):
        self.slots: dict[str, tuple[int, tuple[int, ...]]] = {}
        off = 0
        for name, shape in specs:
            n = int(math.prod(shape)) if len(shape) else 1
            self.slots[name] = (off, tuple(shape))
            off += (n + 15) // 16 * 16
        self.numel = off
        self.data = torch.zeros(max(off, 16), device=device, dtype=dtype)

    def view(self, name: str, buf: torch.Tensor | None = None) -> torch.Tensor:
        off, shape = self.slots[name]
        n = int(math.prod(shape)) if len(shape) else 1
        return (self.data if buf is None else buf)[off:off + n].view(shape)

    def slot(self, name: str, buf: torch.Tensor | None = None, pad_to: int = 16) -> torch.Tensor:
        """1-D view of the whole padded slot (bias vectors read up to the padded channel count)."""
        off, shape = self.slots[name]
        n = int(math.prod(shape)) if len(shape) else 1
        return (self.data if buf is None else buf)[off:off + (n + pad_to - 1) // pad_to * pad_to]

    def like(self) -> torch.Tensor:
        return torch.zeros_like(self.data)


# ---------------------------------------------------------------------------------------------- architecture tables
def mlp_param_specs(prefix: str, cin: int, hidden: int, cout: int, i0="0", i1="1", i3="3"):
    """Linear -> BatchNorm1d -> ReLU -> Linear (r21d_byol.py:232-257,276-291) in registration order."""
    return [(f"{prefix}.{i0}.weight", (hidden, cin)), (f"{prefix}.{i0}.bias", (hidden,)),
            (f"{prefix}.{i1}.weight", (hidden,)), (f"{prefix}.{i1}.bias", (hidden,)),
            (f"{prefix}.{i3}.weight", (cout, hidden)), (f"{prefix}.{i3}.bias", (cout,))]


def stconv_param_specs(prefix: str, cin: int, cout: int, k):
    mid = intermed_channels(cin, cout, k)
    return [(f"{prefix}.spatial_conv.weight", (mid, cin, 1, k[1], k[2])),
            (f"{prefix}.bn.weight", (mid,)), (f"{prefix}.bn.bias", (mid,)),
            (f"{prefix}.temporal_conv.weight", (cout, mid, k[0], 1, 1))]


STAGES = (("conv2", 64, 64, False), ("conv3", 64, 128, True), ("conv4", 128, 256, True), ("conv5", 256, 512, True))


def backbone_param_specs(prefix: str, project: bool = True):
    """R2Plus1DNet((1,1,1,1)) parameters in registration order (SURVEY.md A.5; r21d_byol.py:184-213,113-139)."""
    s = stconv_param_specs(f"{prefix}.conv1", 3, 64, (3, 7, 7))
    s += [(f"{prefix}.bn1.weight", (64,)), (f"{prefix}.bn1.bias", (64,))]
    for stage, cin, cout, down in STAGES:
        b = f"{prefix}.{stage}.block1"
        if down:
            s += stconv_param_specs(b + ".downsampleconv", cin, cout, (1, 1, 1))
            s += [(b + ".downsamplebn.weight", (cout,)), (b + ".downsamplebn.bias", (cout,))]
        s += stconv_param_specs(b + ".conv1", cin, cout, (3, 3, 3))
        s += [(b + ".bn1.weight", (cout,)), (b + ".bn1.bias", (cout,))]
        s += stconv_param_specs(b + ".conv2", cout, cout, (3, 3, 3))
        s += [(b + ".bn2.weight", (cout,)), (b + ".bn2.bias", (cout,))]
    if project:
        s += mlp_param_specs(f"{prefix}.project.net", 512, 4096, 512)
    return s


def trainable_param_specs():
    s = backbone_param_specs("online_net")
    s += mlp_param_specs("predictor.net", 512, 4096, 512)
    s += mlp_param_specs("overlap_spa", 1024, 1024, 5)
    s += mlp_param_specs("overlap_tem", 1024, 1024, 5)
    s += mlp_param_specs("pb_cls", 512, 512, 5)
    s += mlp_param_specs("rotate_cls", 512, 512, 5)
    return s


def bn_buffer_specs(param_specs):
    """running_mean / running_var for every BatchNorm (a 1-D `.weight` whose sibling `.bias` is also 1-D and whose
    module is not a Linear: identified by the absence of a 2-D/5-D weight under the same module name)."""
    out = []
    for name, shape in param_specs:
        if name.endswith(".weight") and len(shape) == 1:
            mod = name[:-len(".weight")]
            out += [(mod + ".running_mean", shape), (mod + ".running_var", shape)]
    return out


# ---------------------------------------------------------------------------------------------- engine
@dataclass
class _Site:
    """One BatchNorm call site: parameters, running buffers and per-step statistics scratch."""
    name: str
    C: int
    gamma: torch.Tensor
    beta: torch.Tensor
    rm: torch.Tensor
    rv: torch.Tensor
    st: "ops.BNState"
    dgamma: torch.Tensor | None = None
    dbeta: torch.Tensor | None = None


class _Timed:
    """A group of tensor-core launches with its algorithmic FLOPs; records CUDA events around the group while the
    engine is in profiling mode (bench.py roofline), otherwise just launches."""

    def __init__(self, eng, kind: str, flops: float, plans, tag: str = ""):
        self.eng, self.kind, self.flops, self.plans, self.tag = eng, kind, flops, list(plans), tag

    def run(self, *args):
        prof = self.eng._prof
        if prof is None:
            for p in self.plans:
                p.run(*args)
            return
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for p in self.plans:
            p.run(*args)
        b.record()
        prof.append((self.kind, self.flops, len(self.plans), a, b, self.tag, ops.kernel_name(self.plans[0])))


class ProgramEngine:
    """What every engine shares: the clip geometry, the flat parameter and BatchNorm-buffer stores, the builders of the
    backbone / MLP launch programs over them, the backward program with its gradient buckets, the bf16 weight packs and
    the CUDA-graph capture of a program.  `B` is the batch (samples; each sample is VIEWS clips, one BatchNorm statistics
    group each).  `specs`: the parameters of the `train` store; `share`: an engine whose parameter and BatchNorm-buffer
    stores this one reads (None: they are allocated here); `grads`: the engine builds a backward program and has a `grad`
    store; `bn_specs`: parameters outside `train` whose BatchNorm running statistics live in `bufs` too."""

    VIEWS = 1          # clips per sample pushed through the backbone = BatchNorm statistics groups
    EVAL_BACKWARD = False   # True: BatchNorm states in the layout of ops.bn_backward_eval (engine_ft.ExplainEngine)

    def __init__(self, B: int, T: int, H: int, W: int, device, specs, *, grads: bool, share=None, bn_specs=(),
                 record: bool = False, overlap: bool = True, bn_sync=None, fuse_apply: bool | None = None,
                 fuse_min_positions: int | None = None, fuse_policy: str | None = None, graph: bool | None = None):
        if H % 2 or W % 4:
            raise ops.L.CstpError("clip height must be even and its width a multiple of 4 (1x7x7 stride-2 stem over packed rows)")
        self.B, self.T, self.H, self.W = B, T, H, W
        self.N = self.VIEWS * B
        self.device = torch.device(device)
        self.record = record
        self.eval_mode = False       # True: BatchNorm uses its running statistics (finetune validation / test)
        # None: per-GPU BatchNorm statistics (what the reference's --sync_bn actually does, SURVEY.md 0.2);
        # a cstp_b200.parallel.BnSync: statistics over every rank of the data-parallel group (north-star SyncBN)
        self.bn_sync = bn_sync
        # Two-stream schedule (CUDA only): the target network's forward runs beside the online network's, and every
        # weight-gradient GEMM runs beside the BatchNorm-backward streaming kernels of the next unit, so HBM-bound and
        # tensor-bound kernels share the machine.  Results are unchanged (same kernels, same reduction orders).
        self.overlap = bool(overlap) and self.device.type == "cuda"
        if self.overlap:
            self._s2 = torch.cuda.Stream(device=self.device)
            self._ev_fwd, self._ev_tgt = torch.cuda.Event(), torch.cuda.Event()
            self._ev_g = [torch.cuda.Event(), torch.cuda.Event()]
            self._ev_wg = [torch.cuda.Event(), torch.cuda.Event()]
            if hasattr(bn_sync, "register_side_stream"):
                bn_sync.register_side_stream(self._s2)
        self._wg_recorded = [False, False]     # has _ev_wg[b] been recorded during the CURRENT backward pass?
        self.use_graph = (USE_GRAPH if graph is None else bool(graph)) and self.device.type == "cuda" and not record
        self._graphs: dict[str, tuple] = {}    # purpose -> (key, CUDA graph, launches per replay): see _captured
        self._ran_eager: set[str] = set()      # purposes whose program has run eagerly once
        self._packed_key = None                # see repack
        self.fuse_apply = FUSE_BN_APPLY if fuse_apply is None else bool(fuse_apply)
        self.fuse_min_positions = FUSE_MIN_POSITIONS if fuse_min_positions is None else int(fuse_min_positions)
        self.fuse_policy = fuse_policy or FUSE_POLICY
        if self.fuse_policy not in ("auto", "all", "none"):
            raise ops.L.CstpError(f"fuse_policy {self.fuse_policy!r}: expected auto, all or none")
        self._pending: dict[int, "ops.BNState"] = {}   # raw tensor address -> BatchNorm state its consumers must apply
        self._pending_act: dict[int, torch.Tensor] = {}   # record mode: the same activations, materialised for the tests
        self.named: dict[str, torch.Tensor] = {}      # name -> activation / gradient tensors (parity tests)
        self.units: list[dict] = []                   # every conv+BN unit in build order (parity tests, profiling)
        self._prof = None                             # list of (kind, flops, launches, ev0, ev1) while profiling

        # ---- flat parameter / gradient / BatchNorm-buffer stores
        if share is None:
            self.train = FlatStore(specs, self.device)
            self.bufs = FlatStore(bn_buffer_specs(list(specs) + list(bn_specs)), self.device)
            for name in self.bufs.slots:
                if name.endswith("running_var"):
                    self.bufs.view(name).fill_(1.0)
        else:
            self.train, self.bufs = share.train, share.bufs
        self.grad = self.train.like() if grads else None

        # ---- scratch shared by all layers
        self._g_numel = 0            # bf16 d(raw) scratch, sized while building
        self._wg_numel = 0           # fp32 wgrad split-K partials scratch
        self._deferred = []          # closures that need the scratch buffers (run after allocation)
        self._dbufs: dict[int, torch.Tensor] = {}
        self._pack_jobs_online = []  # (param view, packed fwd, packed dgrad or None)
        self._pack_jobs_target = []

        self.fwd_online: list = []
        self.fwd_target: list = []
        self.fwd_heads: list = []
        self.bwd: list = []          # executed in order (already reversed while building)

        # ---- inputs
        # stem input: the seven kw taps x three channels of every output column, two frame rows per pixel (ops.stem_pack)
        self.stem_rows = torch.zeros(self.N, T, H // 2, W // 2, ops.STEM_CHANNELS, device=self.device, dtype=ACT_DTYPE)

    # ------------------------------------------------------------------------------------------ helpers
    def _act(self, *shape) -> torch.Tensor:
        return torch.zeros(*shape, device=self.device, dtype=ACT_DTYPE)

    def _dbuf(self, t: torch.Tensor) -> torch.Tensor:
        """Gradient buffer of an activation tensor (keyed by storage address so views share it)."""
        k = t.data_ptr()
        if k not in self._dbufs:
            self._dbufs[k] = torch.zeros_like(t)
        return self._dbufs[k].view(t.shape)

    def _rec(self, name: str, t: torch.Tensor) -> None:
        if self.record:
            self.named[name] = t

    def _site(self, store: FlatStore, grads: bool, name: str, C: int, groups: int, rows_per_group: int) -> _Site:
        st = ops.BNState.alloc(C, pad16(C), groups, rows_per_group, self.device, backward=grads,
                               eval_backward=self.EVAL_BACKWARD)
        return _Site(name, C, store.view(name + ".weight"), store.view(name + ".bias"),
                     self.bufs.view(name + ".running_mean"), self.bufs.view(name + ".running_var"), st,
                     store.view(name + ".weight", self.grad) if grads else None,
                     store.view(name + ".bias", self.grad) if grads else None)

    def _packed(self, store: FlatStore, name: str, grads: bool, rows_pad: int | None = None, stem: bool = False,
                forward: bool = True):
        """bf16 packed forward (and dgrad-transposed) copies of a conv / linear weight; registers the re-pack job.
        stem: the (Cout, 3, 1, 7, 7) weight in the layout of the packed stem row pairs -- four taps of 64 (hpar, kw, c)
        channels (include/cstp_b200.h cstp_pack_weight transpose = 2); it has no dgrad copy.  forward=False: only the
        dgrad copy (a weight whose forward copy another call registered); (None, wt) is returned."""
        w = store.view(name)
        cout, cin = w.shape[0], w.shape[1]
        taps = w.numel() // (cout * cin)
        if stem:
            assert not grads
            cin, taps = ops.STEM_CHANNELS, 4
        wp = None
        if forward:
            wp = torch.zeros(rows_pad or pad16(cout), taps * pad64(pad16(cin)), device=self.device, dtype=ACT_DTYPE)
        wt = None
        if grads:
            wt = torch.zeros(pad16(cin), taps * pad64(pad16(cout)), device=self.device, dtype=ACT_DTYPE)
        (self._pack_jobs_online if store is self.train else self._pack_jobs_target).append((w, wp, wt, 2 if stem else 0))
        return wp, wt

    def _bn_forward(self, raw, site: _Site, fused_blocks: int = 0):
        """BatchNorm forward of `site` over raw: in eval mode (model.eval()) the affine map of the running statistics,
        nothing is updated; otherwise the batch statistics, which also update the running buffers."""
        if self.eval_mode:
            ops.bn_eval_coeffs(site.st, site.gamma, site.beta, site.rm, site.rv, BN_EPS)
        else:
            ops.bn_forward_stats(raw, site.st, site.gamma, site.beta, site.rm, site.rv, BN_EPS, BN_MOMENTUM,
                                 fused_blocks=fused_blocks, sync=self.bn_sync)

    def _captured(self, purpose: str, key, body) -> None:
        """Runs body() -- a program that reads and writes engine-owned buffers only -- eagerly the first time this engine
        runs a program for `purpose` (one-time kernel attributes, NCCL / peer-memory channel set-up), captures it into a
        CUDA graph on the next call and replays that graph from then on.  Another `key` captures again; each purpose keeps
        one graph.  Inputs are written into the static buffers body() reads before the call, outside the graph."""
        held = self._graphs.get(purpose)
        if held is not None and held[0] == key:
            held[1].replay()
            ops.note_replayed(held[2])
            return
        if purpose not in self._ran_eager or not self.use_graph:
            self._ran_eager.add(purpose)
            body()
            return
        torch.cuda.synchronize(self.device)
        before = ops.launch_count()
        g = torch.cuda.CUDAGraph()
        try:
            # thread_local: NCCL's watchdog thread and the data loader's copy stream keep issuing CUDA calls meanwhile
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                body()
        except Exception as e:          # e.g. a collective backend that cannot be captured: stay eager, say so once
            import warnings
            warnings.warn(f"cstp_b200: CUDA-graph capture of the {purpose} program failed ({e!r}); running eagerly")
            self.use_graph = False
            torch.cuda.synchronize(self.device)
            body()
            return
        launches = ops.launch_count() - before
        self._graphs[purpose] = (key, g, launches)
        ops.note_replayed(-launches)       # the capture pass counted launches that did not run
        g.replay()
        ops.note_replayed(launches)

    def _forward_program(self):
        for op in self.fwd_online:
            op()

    # ------------------------------------------------------------------------------------------ conv + BN unit
    def _conv_bn(self, prog, store, grads, x, wname, bnname, geom: ConvGeom, cin, cout, *, relu=True, res=None,
                 res_site=None, apply=True, tag="", skip_dgrad=False, stem=False):
        """raw = conv(x); BN statistics; act = [relu](bn(raw) [+ res]).  Returns (raw, act, site, unit); the backward
        closure of the unit is built by _unit_backward.

        Plain BatchNorm -> ReLU outputs (no shortcut) are NOT materialised when self.fuse_apply: the returned `act` is then
        the raw tensor itself, registered in self._pending with the BatchNorm state its consumers have to apply -- the next
        convolution's forward and weight-gradient kernels through their operand prologue, a residual add through
        bn_apply's res_relu mode, the ReLU mask of the backward pass from raw (it always was)."""
        N, T, H, W, _ = x.shape
        To, Ho, Wo = geom.out_dims(T, H, W)
        Cop = pad16(cout)
        raw = self._act(N, To, Ho, Wo, Cop)
        pro = self._pending.get(x.data_ptr())         # x is a raw tensor whose BatchNorm + ReLU we apply on the way in
        defer = (apply and relu and res is None and self.fuse_apply and self.fuse_policy != "none"
                 and Ho * Wo >= self.fuse_min_positions
                 and (self.fuse_policy == "all" or not grads or geom.kernel[0] == 1))
        keep_act = apply and (not defer or self.record)          # parity tests still look at every activation
        act = self._act(N, To, Ho, Wo, Cop) if keep_act else None
        wp, wt = self._packed(store, wname, grads and not skip_dgrad, stem=stem)
        rows = N * To * Ho * Wo
        flops = 2.0 * rows * cout * cin * (49 if stem else geom.taps)     # algorithmic: the stem is 3 channels x 1x7x7
        site = self._site(store, grads, bnname, cout, self.VIEWS, rows // self.VIEWS)
        cplan = ops.conv_fwd_plan(x, wp, raw, geom, stats=site.st, prologue=pro)
        plan = _Timed(self, "conv_fwd", flops, [cplan], tag)
        fused = getattr(cplan, "stat_blocks", 0)   # > 0: the conv epilogue already wrote the BatchNorm statistics partials
        res_pro = self._pending.get(res.data_ptr()) if res is not None else None
        res_state = res_site.st if res_site else res_pro

        def fwd():
            plan.run()
            self._bn_forward(raw, site, fused)
            if keep_act:
                ops.bn_apply(raw, site.st, act, relu=relu, res=res, res_state=res_state, res_relu=res_pro is not None)
        prog.append(fwd)
        self._rec(tag + ".raw", raw)
        if act is not None:
            self._rec(tag + ".act", act)
        unit = dict(x=x, raw=raw, act=act, site=site, relu=relu, geom=geom, wname=wname, cin=cin, cout=cout, wt=wt,
                    skip_dgrad=skip_dgrad, tag=tag, flops=flops, bnname=bnname, res=res, res_site=res_site,
                    stem=stem, grads=grads, pro=pro, deferred=defer,
                    # what the tensor cores really consume, as materialised tensors (record mode; parity tests)
                    x_act=self._pending_act.get(x.data_ptr(), x).view(x.shape),
                    res_act=self._pending_act.get(res.data_ptr(), res).view(res.shape) if res is not None else None)
        self.units.append(unit)
        self._g_numel = max(self._g_numel, raw.numel())
        out = act
        if defer:
            self._pending[raw.data_ptr()] = site.st
            if act is not None:
                self._pending_act[raw.data_ptr()] = act
            out = raw
        return raw, out, site, unit

    def _unit_backward(self, unit, d_out, *, act_for_mask, dz=None, dx_accumulate=False, eval_dgrad=False):
        """Backward closure of one conv+BN unit: BN backward -> wgrad -> dgrad (see _conv_bn).  eval_dgrad: the eval-mode,
        data-gradient-only flavour (engine_ft.ExplainEngine): the derivative of the running-statistics BatchNorm map
        (ops.bn_backward_eval), then dgrad with a transposed weight packed here; no weight or BatchNorm-parameter
        gradient."""
        x, raw, site, geom = unit["x"], unit["raw"], unit["site"], unit["geom"]
        dw = self.train.view(unit["wname"], self.grad)
        wt = unit["wt"]
        if eval_dgrad and not unit["skip_dgrad"]:
            wt = self._packed(self.train, unit["wname"], True, forward=False)[1]
        holder = {}

        def prepare():
            g = self._gbufs[holder["gbuf"]][:raw.numel()].view(raw.shape)
            holder["g"] = g
            if not eval_dgrad:
                holder["wg"] = _Timed(self, "wgrad", unit["flops"],
                                      [ops.wgrad_plan(x, g, geom, unit["cout"], ops.STEM_CHANNELS if unit["stem"] else unit["cin"],
                                                      self._wg, prologue=unit["pro"], layout=1 if unit["stem"] else 0)],
                                      unit["tag"])
            if not unit["skip_dgrad"]:
                dx = self._dbuf(x)
                plans, covers = ops.conv_dgrad_plans(g, wt, dx, geom, accumulate=dx_accumulate)
                holder["dg"] = _Timed(self, "conv_dgrad", unit["flops"], plans, unit["tag"])
                holder["zero"], holder["dx"] = (not covers and not dx_accumulate), dx
                self._rec(unit["tag"] + ".dx", dx)
        self._deferred.append(prepare)
        if not eval_dgrad:
            self._wg_numel = max(self._wg_numel, self._wgrad_need(x, raw, geom))

        self._rec(unit["tag"] + ".d_out", d_out)
        # plain BN -> ReLU units recompute the mask from raw; block outputs (residual in the pre-activation) read act
        from_raw = act_for_mask is not None and unit["relu"] and unit["res"] is None

        def bwd():
            g = holder["g"]
            if eval_dgrad:
                ops.bn_backward_eval(d_out, act_for_mask, raw, site.st, g, dz=dz, mask_from_raw=from_raw)
            else:
                if self.overlap and self._prof is None and self._wg_recorded[holder["gbuf"]]:
                    # the weight-gradient GEMM that last read this d(raw) buffer (two units ago) must have finished
                    torch.cuda.current_stream().wait_event(self._ev_wg[holder["gbuf"]])
                ops.bn_backward(d_out, act_for_mask, raw, site.st, site.gamma, site.dgamma, site.dbeta, g, dz=dz,
                                mask_from_raw=from_raw, sync=self.bn_sync)
            if self.record:      # parity tests: the shared d(raw) scratch is overwritten by a later unit
                self.named[unit["tag"] + ".g"] = g.clone()
            if eval_dgrad:       # no weight gradient
                pass
            elif self.overlap and self._prof is None:
                b = holder["gbuf"]
                main = torch.cuda.current_stream()
                self._ev_g[b].record(main)
                with torch.cuda.stream(self._s2):
                    self._s2.wait_event(self._ev_g[b])
                    holder["wg"].run(dw)
                    self._ev_wg[b].record(self._s2)
                    self._wg_recorded[b] = True
            else:
                holder["wg"].run(dw)
            if not unit["skip_dgrad"]:
                if holder["zero"]:
                    holder["dx"].zero_()
                holder["dg"].run()
        bwd.holder = holder
        bwd.writes = [] if eval_dgrad else [unit["wname"], unit["bnname"] + ".weight", unit["bnname"] + ".bias"]
        return bwd

    @staticmethod
    def _wgrad_need(x, raw, geom) -> int:
        """Upper bound of the split-K partials (floats) ops.wgrad_plan will need for this layer."""
        return ops.wgrad_partials_need(tuple(x.shape), tuple(raw.shape), geom)

    # ------------------------------------------------------------------------------------------ backbone
    DGRAD_LEVELS = ("input", "conv1") + tuple(s[0] for s in STAGES)

    def _backbone(self, prog, store, prefix, grads, tag, dgrad_to: str | None = None):
        """R2Plus1DNet.forward (r21d_byol.py:215-229) over both views.  Returns (last block act, backward closures in
        forward order).  dgrad_to (without grads): the closures are the eval-mode, data-gradient-only flavour
        (_unit_backward eval_dgrad) of the parts above that level of DGRAD_LEVELS -- "conv5": none, "conv3": the conv4 and
        conv5 blocks, "input": every unit down to the stem's d(raw)."""
        N, T = self.N, self.T
        Ho, Wo = self.H // 2, self.W // 2
        bw: list = []

        def builder(level):
            if grads:
                return self._unit_backward
            if dgrad_to is not None and self.DGRAD_LEVELS.index(level) > self.DGRAD_LEVELS.index(dgrad_to):
                return lambda *a, **k: self._unit_backward(*a, eval_dgrad=True, **k)
            return None
        ub = builder("conv1")
        # stem spatial 1x7x7 s(1,2,2) p(0,3,3) (r21d_byol.py:198): a four-tap stride-1 implicit GEMM over packed row pairs,
        # whose 64 channels hold the (kw, c) taps of every output column for two frame rows -- no im2col matrix in HBM
        _, a0, site, u = self._conv_bn(prog, store, grads, self.stem_rows, f"{prefix}.conv1.spatial_conv.weight",
                                       f"{prefix}.conv1.bn", ops.STEM_GEOM, 3, 83, tag=f"{tag}.conv1.spatial",
                                       skip_dgrad=True, stem=True)
        assert tuple(a0.shape[:4]) == (N, T, Ho, Wo)
        if ub is not None:
            bw.append(ub(u, self._dbuf(a0), act_for_mask=a0))
        raw, x, site, u = self._conv_bn(prog, store, grads, a0, f"{prefix}.conv1.temporal_conv.weight", f"{prefix}.bn1",
                                        ConvGeom((3, 1, 1), (1, 1, 1), (1, 0, 0)), 83, 64, tag=f"{tag}.conv1.temporal")
        if ub is not None:
            bw.append(ub(u, self._dbuf(x), act_for_mask=x))
        for stage, cin, cout, down in STAGES:
            x = self._block(prog, store, f"{prefix}.{stage}.block1", grads, x, cin, cout, down, bw,
                            f"{tag}.{stage}.block1", unit_backward=builder(stage))
        return x, bw

    def _block(self, prog, store, pre, grads, xin, cin, cout, down, bw, tag, unit_backward=None):
        """SpatioTemporalResBlock.forward (r21d_byol.py:141-148).  unit_backward: the builder of the backward closures
        appended to bw (None: _unit_backward with grads, no closures without)."""
        s = 2 if down else 1
        mid1 = intermed_channels(cin, cout, (3, 3, 3))
        mid2 = intermed_channels(cout, cout, (3, 3, 3))
        sp = lambda st: ConvGeom((1, 3, 3), (1, st, st), (0, 1, 1))
        tp = lambda st: ConvGeom((3, 1, 1), (st, 1, 1), (1, 0, 0))
        _, a, _, u1 = self._conv_bn(prog, store, grads, xin, f"{pre}.conv1.spatial_conv.weight", f"{pre}.conv1.bn", sp(s),
                                    cin, mid1, tag=f"{tag}.conv1.spatial")
        _, b, _, u2 = self._conv_bn(prog, store, grads, a, f"{pre}.conv1.temporal_conv.weight", f"{pre}.bn1", tp(s),
                                    mid1, cout, tag=f"{tag}.conv1.temporal")
        _, c, _, u3 = self._conv_bn(prog, store, grads, b, f"{pre}.conv2.spatial_conv.weight", f"{pre}.conv2.bn", sp(1),
                                    cout, mid2, tag=f"{tag}.conv2.spatial")
        if down:
            midd = intermed_channels(cin, cout, (1, 1, 1))
            _, d1, _, u5 = self._conv_bn(prog, store, grads, xin, f"{pre}.downsampleconv.spatial_conv.weight",
                                         f"{pre}.downsampleconv.bn", ConvGeom((1, 1, 1), (1, 2, 2)), cin, midd,
                                         tag=f"{tag}.downsampleconv.spatial")
            raw_ds, _, site_ds, u6 = self._conv_bn(prog, store, grads, d1, f"{pre}.downsampleconv.temporal_conv.weight",
                                                   f"{pre}.downsamplebn", ConvGeom((1, 1, 1), (2, 1, 1)), midd, cout,
                                                   relu=False, apply=False, tag=f"{tag}.downsampleconv.temporal")
            _, out, _, u4 = self._conv_bn(prog, store, grads, c, f"{pre}.conv2.temporal_conv.weight", f"{pre}.bn2", tp(1),
                                          mid2, cout, relu=True, res=raw_ds, res_site=site_ds,
                                          tag=f"{tag}.conv2.temporal")
        else:
            _, out, _, u4 = self._conv_bn(prog, store, grads, c, f"{pre}.conv2.temporal_conv.weight", f"{pre}.bn2", tp(1),
                                          mid2, cout, relu=True, res=xin, tag=f"{tag}.conv2.temporal")
        self._rec(tag + ".out", out)
        ub = unit_backward or (self._unit_backward if grads else None)
        if ub is not None:
            d_out = self._dbuf(out)
            if down:
                dz = self._act(*out.shape)          # masked upstream gradient, shared by bn2 and downsamplebn
                self._rec(tag + ".dz", dz)
                # forward order: u1 u2 u3 u5 u6 u4  -> reversed at run time
                bw.append(ub(u1, self._dbuf(a), act_for_mask=a))                 # writes d(xin)
                bw.append(ub(u2, self._dbuf(b), act_for_mask=b))
                bw.append(ub(u3, self._dbuf(c), act_for_mask=c))
                # run order is reversed, so u5/u6 must come BEFORE u1 in the list to run AFTER it: they accumulate
                # into d(xin) that u1 has overwritten.  Insert them ahead of u1.
                k = len(bw) - 3
                bw.insert(k, ub(u5, self._dbuf(d1), act_for_mask=d1, dx_accumulate=True))
                bw.insert(k + 1, ub(u6, dz, act_for_mask=None))
                bw.append(ub(u4, d_out, act_for_mask=out, dz=dz))
            else:
                # bn2 backward writes the masked upstream gradient straight into d(xin) (identity shortcut); the conv1
                # spatial dgrad then accumulates into it.
                bw.append(ub(u1, self._dbuf(a), act_for_mask=a, dx_accumulate=True))
                bw.append(ub(u2, self._dbuf(b), act_for_mask=b))
                bw.append(ub(u3, self._dbuf(c), act_for_mask=c))
                bw.append(ub(u4, d_out, act_for_mask=out, dz=self._dbuf(xin)))
        return out

    # ------------------------------------------------------------------------------------------ MLP heads
    def _mlp(self, prog, store, grads, x, pre, cin, hidden, cout, groups, *, names=("0", "1", "3"), out_bf16=False,
             tag=""):
        """Linear -> BatchNorm1d -> ReLU -> Linear.  x: bf16 [rows][pad16(cin)].  Returns dict with out_f32 [rows][Op]
        (+ out_bf16) and, when `grads`, a backward factory taking (d_out fp32 [rows][Op], scale_dev, dx_f32, accumulate)."""
        i0, i1, i3 = names
        rows = x.shape[0]
        Hp, Op = pad16(hidden), pad16(cout)
        raw = self._act(rows, Hp)
        h = self._act(rows, Hp)
        outf = torch.zeros(rows, Op, device=self.device, dtype=torch.float32)
        outb = self._act(rows, Op) if out_bf16 else None
        w0, w0t = self._packed(store, f"{pre}.{i0}.weight", grads)
        w3, w3t = self._packed(store, f"{pre}.{i3}.weight", grads)
        b0 = store.slot(f"{pre}.{i0}.bias")
        b3 = store.slot(f"{pre}.{i3}.bias")
        p0 = ops.linear_plan(x, w0, raw, bias=b0)
        p3 = ops.linear_plan(h, w3, outb, out_f32=outf, bias=b3)
        site = self._site(store, grads, f"{pre}.{i1}", hidden, groups, rows // groups)

        def fwd():
            p0.run()
            self._bn_forward(raw, site)
            ops.bn_apply(raw, site.st, h, relu=True)
            p3.run()
        prog.append(fwd)
        self._rec(tag + ".x", x)
        self._rec(tag + ".raw", raw)
        self._rec(tag + ".h", h)
        self._rec(tag + ".out", outf)
        res = dict(out_f32=outf, out_bf16=outb, site=site)
        if not grads:
            return res
        g_out = self._act(rows, Op)
        d_h = self._act(rows, Hp)
        g_h = self._act(rows, Hp)
        dW0 = store.view(f"{pre}.{i0}.weight", self.grad)
        dW3 = store.view(f"{pre}.{i3}.weight", self.grad)
        db0 = store.view(f"{pre}.{i0}.bias", self.grad)
        db3 = store.view(f"{pre}.{i3}.bias", self.grad)
        g1 = ConvGeom((1, 1, 1))
        x5, h5 = x.view(1, 1, 1, rows, -1), h.view(1, 1, 1, rows, Hp)
        go5, gh5 = g_out.view(1, 1, 1, rows, Op), g_h.view(1, 1, 1, rows, Hp)
        self._rec(tag + ".g_out", g_out)
        self._rec(tag + ".d_h", d_h)
        self._rec(tag + ".g_h", g_h)
        self._wg_numel = max(self._wg_numel, self._wgrad_need(h5, go5, g1), self._wgrad_need(x5, gh5, g1))
        holder = {}

        def make_backward(d_out, scale_dev, dx_f32, accumulate):
            """d_out fp32 [rows][Op] (optionally scaled by the device scalar) -> parameter grads and dx_f32 [rows][Cip]."""
            pd_h = ops.linear_plan(g_out, w3t, d_h)
            pd_x = ops.linear_plan(g_h, w0t, None, out_f32=dx_f32, accumulate=accumulate) if dx_f32 is not None else None

            def prepare():
                holder["wg3"] = ops.wgrad_plan(h5, go5, g1, cout, hidden, self._wg)
                holder["wg0"] = ops.wgrad_plan(x5, gh5, g1, hidden, cin, self._wg)
            self._deferred.append(prepare)

            self._rec(tag + ".dx", dx_f32)
            self._rec(tag + ".dx_accumulate", accumulate)

            def bwd():
                ops.cast_pad(d_out, g_out, cols=cout, scale_dev=scale_dev)
                ops.colsum(g_out, cout, db3)
                holder["wg3"].run(dW3)
                pd_h.run()
                ops.bn_backward(d_h, h, raw, site.st, site.gamma, site.dgamma, site.dbeta, g_h, mask_from_raw=True,
                                sync=self.bn_sync)
                ops.colsum(g_h, hidden, db0)
                holder["wg0"].run(dW0)
                if pd_x is not None:
                    pd_x.run()
            bwd.writes = [f"{pre}.{i0}.weight", f"{pre}.{i0}.bias", f"{pre}.{i1}.weight", f"{pre}.{i1}.bias",
                          f"{pre}.{i3}.weight", f"{pre}.{i3}.bias"]
            return bwd
        res["make_backward"] = make_backward
        return res

    # ------------------------------------------------------------------------------------------ build
    def _finish_build(self):
        """Shared scratch + deferred plan creation, once every forward / backward closure exists."""
        f32 = dict(device=self.device, dtype=torch.float32)
        # d(raw) scratch: two buffers, alternating in RUN order, so that a unit's weight-gradient GEMM (side stream) can
        # still read its d(raw) while the next unit's BatchNorm backward writes the other buffer
        turn = 0
        for op in self.bwd:
            h = getattr(op, "holder", None)
            if h is not None:
                h["gbuf"] = turn
                turn ^= 1 if self.overlap else 0
        self._gbufs = [self._act(self._g_numel)]
        self._gbufs.append(self._act(self._g_numel) if self.overlap else self._gbufs[0])
        self._wg = torch.zeros(self._wg_numel, **f32)
        for fn in self._deferred:
            fn()
        self._deferred.clear()
        self._plan_grad_buckets()

    GRAD_BUCKET_MIN = 3_000_000      # elements (12 MB of fp32): below this an all-reduce is latency, not bandwidth

    def _plan_grad_buckets(self):
        """Where the data-parallel gradient all-reduce can start before the backward pass has finished.  The flat gradient
        buffer is laid out in registration order and the backward program runs (roughly) in the reverse order, so after
        closure i every slot at or above a low-water mark is final: {closure index: (lo, hi)} hands the newly finished
        tail [lo, hi) to the communication stream whenever it has grown past GRAD_BUCKET_MIN; the last closure sends the
        rest.  (DDP's bucketed hooks, models/model.py:97-103, on one contiguous buffer.)"""
        slots = self.train.slots
        order = sorted(slots.items(), key=lambda kv: kv[1][0])           # (name, (offset, shape)) by offset
        remaining = {n: 0 for n in slots}
        for op in self.bwd:
            for n in getattr(op, "writes", ()):
                if n in remaining:
                    remaining[n] += 1
        never = {n for n, c in remaining.items() if c == 0}              # parameters no closure writes (frozen backbone)
        self._grad_buckets, sent = {}, self.train.numel
        for i, op in enumerate(self.bwd):
            for n in getattr(op, "writes", ()):
                if n in remaining:
                    remaining[n] -= 1
            mark = self.train.numel
            for n, (off, _) in reversed(order):
                if remaining[n] > 0 and n not in never:
                    break
                mark = off
            last = i == len(self.bwd) - 1
            if last:
                mark = 0
            if sent - mark >= (1 if last else self.GRAD_BUCKET_MIN):
                self._grad_buckets[i] = (mark, sent)
                sent = mark
        if self.device.type == "cuda":
            self._bucket_events = {i: torch.cuda.Event() for i in self._grad_buckets}

    # ------------------------------------------------------------------------------------------ programs
    def _pack_list(self, jobs):
        flat = []
        for w, wp, wt, mode in jobs:
            if wp is not None:
                flat.append((w, wp, mode))
            if wt is not None:
                flat.append((w, wt, 1))
        return ops.PackList(flat, self.device)

    def pack_online(self):
        """fp32 master weights -> bf16 tensor-core copies (forward and dgrad-transposed), one launch for the network."""
        if getattr(self, "_pl_online", None) is None:
            self._pl_online = self._pack_list(self._pack_jobs_online)
        self._pl_online.run()

    def pack_target(self):
        if getattr(self, "_pl_target", None) is None:
            self._pl_target = self._pack_list(self._pack_jobs_target)
        self._pl_target.run()

    def repack(self, key, packed: bool = False) -> None:
        """Re-packs the bf16 weights unless they were last packed at `key`, the caller's version of the fp32 parameters
        (which other engines may share and change); packed=True only records that they are current at `key` (the
        optimiser step that changed them re-packed them)."""
        if key != self._packed_key and not packed:
            self.pack_online()
        self._packed_key = key

    def backward(self, grad_sync=None):
        """Runs the backward program.  `grad_sync` (a parallel.GradSync): finished tails of the flat gradient buffer are
        all-reduced on its communication stream while the rest of the backward pass still runs (call grad_sync.finish()
        before the optimiser); returns True when the buffer was handed over that way."""
        bucketed = grad_sync is not None and hasattr(grad_sync, "bucket") and self._prof is None
        side = self.overlap and self._prof is None
        self._wg_recorded = [False, False]
        for i, op in enumerate(self.bwd):
            op()
            if bucketed and i in self._grad_buckets:
                lo, hi = self._grad_buckets[i]
                events = []
                if self.device.type == "cuda":
                    ev = self._bucket_events[i]
                    ev.record()
                    events = [ev] + ([e for e, r in zip(self._ev_wg, self._wg_recorded) if r] if side else [])
                grad_sync.bucket(self.grad[lo:hi], events)
        if side:
            main = torch.cuda.current_stream()
            for e, r in zip(self._ev_wg, self._wg_recorded):
                if r:
                    main.wait_event(e)
        return bucketed


class OptimizerEngine(ProgramEngine):
    """An engine that steps an optimiser over its whole flat parameter buffer (the pretraining and finetune engines):
    global-norm clip + SGD momentum or Adam / AdamW, with their state mirroring `train`, then the bf16 re-pack."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, grads=True, **kwargs)
        f32 = dict(device=self.device, dtype=torch.float32)
        self.mom = self.train.like()
        self.first_step = True       # no optimiser state yet (SGD momentum / Adam moments)
        self.optim_kind = "sgd"      # the optimiser the state belongs to (OPTIMIZERS)
        self.adam_step = 0           # Adam / AdamW steps taken (torch's per-parameter `step`)
        self.exp_avg = self.exp_avg_sq = self.adam_hyper = None
        self.norm_out = torch.zeros(2, **f32)
        self.sgd_ws = torch.zeros(2048, **f32)
        # the hyper-parameters of a captured SGD step {lr, momentum, wd, max_norm, do_clip, first_step}
        # (cstp_sgd_clip_step_dev)
        self.hyper = torch.zeros(8, **f32)
        self._hyper_host = None

    def select_optimizer(self, kind: str) -> None:
        """Binds the optimiser `kind` (OPTIMIZERS) for the next step.  Adam's state buffers (exp_avg / exp_avg_sq mirrors
        of the trainable buffer) are allocated when Adam first runs, so an SGD run holds nothing extra.  Optimiser state
        belongs to one kind: asking for another while it exists raises ValueError."""
        if kind not in OPTIMIZERS:
            raise ValueError(f"optimizer {kind!r}: expected one of {OPTIMIZERS}")
        if kind != self.optim_kind and not self.first_step:
            raise ValueError(f"the engine holds {self.optim_kind} optimiser state; it cannot continue as {kind}")
        self.optim_kind = kind
        if kind == "sgd":
            return
        if self.exp_avg is None:
            self.exp_avg, self.exp_avg_sq = self.train.like(), self.train.like()
            self.adam_hyper = torch.zeros(len(ops.L.AdamHyper._fields_), device=self.device, dtype=torch.float32)
        elif self.first_step:
            self.exp_avg.zero_()
            self.exp_avg_sq.zero_()
        if self.first_step:
            self.adam_step = 0

    def _next_adam(self, lr, betas, eps, wd, max_norm, clip) -> tuple:
        self.adam_step += 1
        return adam_scalars(self.adam_step, lr, betas, eps, wd, self.optim_kind == "adamw", max_norm, clip)

    def take_optimizer_state(self, other: "StepEngine") -> None:
        """Continues the optimiser of `other`, an engine of another batch geometry over the same parameter layout that is
        about to be dropped (its Adam moments are taken over, not copied)."""
        self.mom.copy_(other.mom)
        self.first_step, self.optim_kind, self.adam_step = other.first_step, other.optim_kind, other.adam_step
        self.exp_avg, self.exp_avg_sq, self.adam_hyper = other.exp_avg, other.exp_avg_sq, other.adam_hyper

    def optimizer_step(self, lr, momentum=0.9, wd=5e-4, max_norm=18.0, clip=True, optimizer="sgd", betas=(0.9, 0.999),
                       eps=1e-8):
        """clip_grad_norm_ + SGD.step (main_byol.py:88-91,229-232), or + Adam / AdamW.step (`momentum` unused), on the flat
        buffers, then re-pack the bf16 weights."""
        self.select_optimizer(optimizer)
        n = self.train.numel
        if optimizer == "sgd":
            ops.sgd_clip_step(self.train.data[:n], self.grad[:n], self.mom[:n], lr, momentum, wd, max_norm, clip,
                              self.first_step, self.norm_out, self.sgd_ws)
        else:
            ops.adam_clip_step(self.train.data[:n], self.grad[:n], self.exp_avg[:n], self.exp_avg_sq[:n],
                               self._next_adam(lr, betas, eps, wd, max_norm, clip), self.norm_out, self.sgd_ws)
        self.first_step = False
        self.pack_online()

    def set_hyper(self, lr, momentum, wd, max_norm, clip) -> None:
        """Writes the optimiser's hyper-parameters (and the first-step flag) into device memory when they changed."""
        h = (float(lr), float(momentum), float(wd), float(max_norm), 1.0 if clip else 0.0, 1.0 if self.first_step else 0.0)
        if h != self._hyper_host:
            self.hyper[:6].copy_(torch.tensor(h, dtype=torch.float32), non_blocking=False)
            self._hyper_host = h

    def set_adam_hyper(self, lr, betas, eps, wd, max_norm, clip) -> None:
        """Writes the scalars of the next Adam / AdamW step into device memory, in stream order ahead of the step (through
        pinned memory, which torch's host allocator keeps until the copy has run: the host does not wait)."""
        h = torch.tensor(self._next_adam(lr, betas, eps, wd, max_norm, clip), dtype=torch.float32)
        self.adam_hyper.copy_(h.pin_memory(), non_blocking=True)


class StepEngine(OptimizerEngine):
    """See the module docstring.  `B` is the per-GPU batch (samples; each sample is two views)."""

    VIEWS = 2

    def __init__(self, B: int, T: int = 16, H: int = 112, W: int = 112, device="cuda", momentum_ema: float = 0.996,
                 record: bool = False, overlap: bool = True, bn_sync=None, fuse_apply: bool | None = None,
                 ntxent: dict | None = None, fuse_min_positions: int | None = None, fuse_policy: str | None = None,
                 graph: bool | None = None, collapse_stats: bool = False):
        target_specs = backbone_param_specs("target_net")
        super().__init__(B, T, H, W, device, trainable_param_specs(), bn_specs=target_specs, record=record,
                         overlap=overlap, bn_sync=bn_sync, fuse_apply=fuse_apply, fuse_min_positions=fuse_min_positions,
                         fuse_policy=fuse_policy, graph=graph)
        self.momentum_ema = momentum_ema
        # optional NT-Xent term on the online projector outputs of the two views (north-star extension: the reference
        # builds NTXentLoss but never calls it, SURVEY.md 0.1): dict(weight, temperature, gather) -- with gather the
        # embeddings of every rank are all-gathered first, so each rank contrasts against the GLOBAL batch
        # (loss/NTXent.py:46-62 with batch_size = opts.batch_size, main_byol.py:191-196)
        self.ntxent = dict(ntxent) if ntxent else None
        self.target = FlatStore(target_specs, self.device)
        self.online_numel = FlatStore(backbone_param_specs("online_net"), "meta").numel
        assert self.online_numel == self.target.numel
        f32 = dict(device=self.device, dtype=torch.float32)
        self.weights5 = torch.tensor([0.1, 1.0, 1.0, 1.0, 1.0], **f32)
        self.losses = torch.zeros(8, **f32)       # [0..5] CE, [6] weighted CE sum, [7] BYOL loss
        # collapse statistics (cstp_repr_stats) of the last forward run with collapse_stats on: [view][REPR_STATS].
        # Changing the flag changes the step program: drop a captured graph first (R21DBYOL.train_step does).
        self.collapse_stats = bool(collapse_stats)
        self.step_stats = torch.zeros(2, len(REPR_STATS), **f32)
        # static integer labels (spa, tem, pb, rot1, rot2) of the captured step
        self.labels_static = tuple(torch.zeros(B, dtype=torch.int64, device=self.device) for _ in range(5))
        self._build()

    @property
    def _graph(self):
        """The captured training step (graphed_step); None until it has been captured."""
        held = self._graphs.get("step")
        return held and held[1]

    # ------------------------------------------------------------------------------------------ build
    def _build(self):
        B, N = self.B, self.N
        f32 = dict(device=self.device, dtype=torch.float32)
        # ---------------- online network + projector + predictor
        x5, bw_backbone = self._backbone(self.fwd_online, self.train, "online_net", True, "online")
        P = x5.shape[1] * x5.shape[2] * x5.shape[3]
        self.feat = torch.zeros(N, 512, **f32)                 # rows [0,B) view 1, [B,2B) view 2
        self.feat_bf = self._act(N, 512)
        self.feat_cat = self._act(B, 1024)                     # cat(feat1, feat2) (r21d_byol.py:374)
        self.fwd_online.append(lambda: (ops.avgpool_fwd(x5, self.feat, self.feat_bf),
                                        ops.avgpool_fwd(x5, None, self.feat_cat, rows_out=B, ld_out=1024)))
        self._rec("online.feat", self.feat)
        proj = self._mlp(self.fwd_online, self.train, True, self.feat_bf, "online_net.project.net", 512, 4096, 512, 2,
                         out_bf16=True, tag="online.project")
        pred = self._mlp(self.fwd_online, self.train, True, proj["out_bf16"], "predictor.net", 512, 4096, 512, 2,
                         tag="predictor")
        self.pred = pred["out_f32"]
        # ---------------- target network (no gradients; its own activations are scratch)
        t5, _ = self._backbone(self.fwd_target, self.target, "target_net", False, "target")
        self.tfeat_bf = self._act(N, 512)
        self.fwd_target.append(lambda: ops.avgpool_fwd(t5, None, self.tfeat_bf))
        tproj = self._mlp(self.fwd_target, self.target, False, self.tfeat_bf, "target_net.project.net", 512, 4096, 512, 2,
                          tag="target.project")
        self.tproj = tproj["out_f32"]
        # ---------------- pretext heads (r21d_byol.py:374-380)
        spa = self._mlp(self.fwd_heads, self.train, True, self.feat_cat, "overlap_spa", 1024, 1024, 5, 1, tag="overlap_spa")
        tem = self._mlp(self.fwd_heads, self.train, True, self.feat_cat, "overlap_tem", 1024, 1024, 5, 1, tag="overlap_tem")
        pb = self._mlp(self.fwd_heads, self.train, True, self.feat_bf, "pb_cls", 512, 512, 5, 2, tag="pb_cls")
        rot = self._mlp(self.fwd_heads, self.train, True, self.feat_bf, "rotate_cls", 512, 512, 5, 2, tag="rotate_cls")
        self.logit_bufs = (spa["out_f32"], tem["out_f32"], pb["out_f32"], rot["out_f32"])
        # views in the reference's return order: spa, tem, pb1, pb2, rot1, rot2 (each [B][16], 5 valid columns)
        self.logits6 = (spa["out_f32"], tem["out_f32"], pb["out_f32"][:B], pb["out_f32"][B:], rot["out_f32"][:B],
                        rot["out_f32"][B:])
        self.dlogit_bufs = tuple(torch.zeros_like(t) for t in self.logit_bufs)
        d = self.dlogit_bufs
        self.dlogits6 = (d[0], d[1], d[2][:B], d[2][B:], d[3][:B], d[3][B:])
        # ---------------- backward program
        self.dpred = torch.zeros(N, 512, **f32)      # dL_byol/dpred for upstream 1 (scaled inside cast_pad)
        self.dproj = torch.zeros(N, 512, **f32)
        self.dfeat = torch.zeros(N, 512, **f32)
        self.dcat = torch.zeros(B, 1024, **f32)
        self.byol_scale = torch.ones(1, **f32)       # d(total)/d(loss_byol) (= loss_weight[0] on the fused path)
        bw = self.bwd
        bw.append(pred["make_backward"](self.dpred, self.byol_scale, self.dproj, False))
        self.proj_out = proj["out_f32"]
        if self.ntxent is not None:
            self._ntxent_setup()
            bw.append(self._ntxent_backward)
        bw.append(proj["make_backward"](self.dproj, None, self.dfeat, False))
        bw.append(pb["make_backward"](d[2], None, self.dfeat, True))
        bw.append(rot["make_backward"](d[3], None, self.dfeat, True))
        bw.append(spa["make_backward"](d[0], None, self.dcat, False))
        bw.append(tem["make_backward"](d[1], None, self.dcat, True))
        d_x5 = self._dbuf(x5)
        bw.append(lambda: ops.avgpool_bwd(self.dfeat, d_x5, dcat=self.dcat))
        bw.extend(reversed(bw_backbone))
        # ---------------- shared scratch + deferred plan creation
        self._finish_build()

    # ------------------------------------------------------------------------------------------ NT-Xent term
    def _ntxent_setup(self):
        import torch.distributed as dist
        o = self.ntxent
        o.setdefault("weight", 1.0)
        o.setdefault("temperature", 0.1)
        gather = bool(o.get("gather", False)) and dist.is_available() and dist.is_initialized()
        self._nx_world = dist.get_world_size() if gather else 1
        self._nx_rank = dist.get_rank() if gather else 0
        B, W = self.B, self._nx_world
        f32 = dict(device=self.device, dtype=torch.float32)
        self._nx_local = torch.zeros(2, B, 512, **f32)           # [zjs = view 2 | zis = view 1] of this rank
        self._nx_all = torch.zeros(W, 2, B, 512, **f32)
        self._nx_z = torch.zeros(2 * W * B, 512, **f32)          # cat(zjs of every rank, zis of every rank): NTXent.py:47
        self._nx_dz = torch.zeros(2 * W * B, 512, **f32)
        self.ntxent_loss = torch.zeros(1, **f32)
        self._nx_ws = torch.empty(ops.ntxent_workspace_floats(2 * W * B, 512), **f32)

    def _ntxent_forward(self):
        """NTXentLoss(zis = projector(view 1), zjs = projector(view 2)) over the (gathered) batch: loss + d(loss)/dz."""
        B, W = self.B, self._nx_world
        p = self.proj_out[:, :512]
        self._nx_local[0].copy_(p[B:])
        self._nx_local[1].copy_(p[:B])
        if W > 1:
            import torch.distributed as dist
            dist.all_gather_into_tensor(self._nx_all.view(W * 2, B, 512), self._nx_local)
            self._nx_z.view(2, W, B, 512).copy_(self._nx_all.permute(1, 0, 2, 3))
        else:
            self._nx_z.view(2, B, 512).copy_(self._nx_local)
        ops.ntxent(self._nx_z, float(self.ntxent["temperature"]), True, self.ntxent_loss, self._nx_dz, self._nx_ws)

    def _ntxent_backward(self):
        """Adds weight * d(NT-Xent)/d(projector output) of this rank's rows to dproj.  Every rank evaluates the same global
        loss, so the local slice carries a factor `world` that the data-parallel gradient mean removes again
        (parallel._AllGather)."""
        B, W, r = self.B, self._nx_world, self._nx_rank
        dz = self._nx_dz.view(2, W, B, 512)
        a = float(self.ntxent["weight"]) * W
        self.dproj[:B, :512].add_(dz[1, r], alpha=a)
        self.dproj[B:, :512].add_(dz[0, r], alpha=a)

    def load_clips(self, x1: torch.Tensor, x2: torch.Tensor):
        """fp32 NCDHW clips (B,3,T,H,W) -> bf16 packed stem rows (shared by the online and target nets)."""
        ops.stem_pack(x1, self.stem_rows[:self.B])
        ops.stem_pack(x2, self.stem_rows[self.B:])

    def ema(self):
        """R21DBYOL._update_target_net (r21d_byol.py:331-337) over the flat buffers, then re-pack the target weights."""
        ops.ema_update(self.target.data[:self.target.numel], self.train.data[:self.online_numel], self.momentum_ema)
        self.pack_target()

    def forward(self, x1, x2, repack_online: bool = False):
        """R21DBYOL.forward(o_type='loss_com') -- r21d_byol.py:357-382.  Fills self.losses[7] (BYOL), self.logits6 and
        self.dpred (gradient of the BYOL loss w.r.t. the predictor output for upstream 1)."""
        if repack_online:
            self.pack_online()
        self.load_clips(x1, x2)
        self._forward_body()

    def _forward_body(self):
        """Everything of forward() behind the input pass: reads only engine-owned buffers (capturable)."""
        if self.overlap and self._prof is None:
            main = torch.cuda.current_stream()
            self._ev_fwd.record(main)
            with torch.cuda.stream(self._s2):
                self._s2.wait_event(self._ev_fwd)
                self.ema()                       # reads the online weights, which nothing writes during the forward
                for op in self.fwd_target:
                    op()
                self._ev_tgt.record(self._s2)
            for op in self.fwd_online:
                op()
            main.wait_event(self._ev_tgt)
        else:
            for op in self.fwd_online:
                op()
            self.ema()
            for op in self.fwd_target:
                op()
        ops.byol_loss(self.pred, self.tproj, self.B, 512, self.losses[7:8], None, self.dpred)
        if self.collapse_stats:           # reads buffers the step writes anyway: nothing else changes
            ops.repr_stats(self.feat, self.proj_out, self.pred, self.tproj, self.B, self.step_stats)
        if self.ntxent is not None:
            self._ntxent_forward()
        for op in self.fwd_heads:
            op()

    def pretext_losses(self, labels5):
        """Six CrossEntropyLoss terms + the --loss_weight sum (main_byol.py:62-73); writes dlogits for backward."""
        spa, tem, pb, r1, r2 = labels5
        ops.pretext_ce(self.logits6, (spa, tem, pb, pb, r1, r2), self.dlogits6, self.B, 5, self.weights5, self.losses)

    # ------------------------------------------------------------------------------------------ captured step
    def _step_body(self, grad_sync, after):
        """forward (behind the input pass) -> pretext losses -> backward (+ gradient all-reduce) -> optimiser -> re-pack,
        on engine-owned buffers only: the program graphed_step captures."""
        self._forward_body()
        self.pretext_losses(self.labels_static)
        if self.backward(grad_sync):
            grad_sync.finish()
        elif grad_sync is not None:
            grad_sync(self.grad)
        n = self.train.numel
        if self.optim_kind == "sgd":
            ops.sgd_clip_step_dev(self.train.data[:n], self.grad[:n], self.mom[:n], self.hyper, self.norm_out, self.sgd_ws)
        else:
            ops.adam_clip_step_dev(self.train.data[:n], self.grad[:n], self.exp_avg[:n], self.exp_avg_sq[:n],
                                   self.adam_hyper, self.norm_out, self.sgd_ws)
        self.pack_online()
        if after is not None:
            after()

    def graphed_step(self, x1, x2, labels, lr, momentum, wd, max_norm, clip, grad_sync=None, after=None, optimizer="sgd",
                     betas=(0.9, 0.999), eps=1e-8):
        """One pretraining step with everything behind the input pass replayed from a CUDA graph.  The first call runs the
        program eagerly (one-time kernel attributes, NCCL / peer-memory channel set-up), the second captures it; inputs
        (clips -> packed stem rows, labels, hyper-parameters) are written into static buffers in front of the graph.
        `after` (device-side bookkeeping of the caller, e.g. num_batches_tracked) is part of the program and must be the
        same callable for the lifetime of a capture; drop_graph() forgets the capture.  Each optimiser kind is a capture of
        its own (Adam / AdamW: the step-dependent scalars are rewritten in device memory before every replay)."""
        self.select_optimizer(optimizer)
        self.load_clips(x1, x2)
        for dst, src in zip(self.labels_static, labels):
            dst.copy_(src)
        if optimizer == "sgd":
            self.set_hyper(lr, momentum, wd, max_norm, clip)
        else:
            self.set_adam_hyper(lr, betas, eps, wd, max_norm, clip)
        self._captured("step", (id(grad_sync), optimizer), lambda: self._step_body(grad_sync, after))
        self.first_step = False

    def drop_graph(self) -> None:
        self._graphs.pop("step", None)

    def profile_tensor_launches(self, x1, x2):
        """Runs one forward + backward with CUDA events around every backbone tensor-core launch group.
        Returns {kind: (ms, algorithmic FLOPs, launches)} for kind in conv_fwd / conv_dgrad / wgrad; the per-group
        records (kind, layer tag, ms, FLOPs, launches, kernel name) are kept in self.last_profile."""
        self._prof = []
        try:
            self.forward(x1, x2)
            self.backward()
            torch.cuda.synchronize()
            out: dict = {}
            self.last_profile = []          # per launch group: (kind, tag, ms, flops, launches)
            for kind, flops, n, a, b, tag, kernel in self._prof:
                ms, fl, cnt = out.get(kind, (0.0, 0.0, 0))
                out[kind] = (ms + a.elapsed_time(b), fl + flops, cnt + n)
                self.last_profile.append((kind, tag, a.elapsed_time(b), flops, n, kernel))
        finally:
            self._prof = None
        return out

    def set_loss_weight(self, w5):
        self.weights5.copy_(torch.tensor([float(v) for v in w5], dtype=torch.float32))
        self.byol_scale.copy_(self.weights5[0:1])
