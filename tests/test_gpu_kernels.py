"""Kernel-family parity through the C ABI on a B200: implicit-GEMM conv forward / dgrad / wgrad at the layer shapes of
R2Plus1DNet (SURVEY.md A.1), linear layers, BatchNorm forward/backward, the stem over packed rows, EMA (bit-exact),
clip + SGD, BYOL and pretext cross-entropy losses -- each against the fp32 torch operator on identical (bf16-rounded)
inputs.
The case bodies live in tools/gpu_kernel_check.py (also usable as a stand-alone bring-up harness)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _exact_fp32_reference():
    old = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old


def _cases(kind):
    from tools.gpu_kernel_check import CASES
    return [n for n, (k, _) in CASES.items() if k == kind]


@pytest.mark.parametrize("name", _cases("conv"))
def test_conv_forward_dgrad_wgrad(name):
    from tools.gpu_kernel_check import run_case
    r = run_case(name)
    assert r["fwd_nan"] == 0 and r["fwd_pad_zero"]
    assert r["fwd_rel"] < 4e-3, r            # bf16 output rounding of an fp32-accumulated sum: ~2^-9 RMS
    assert r["dgrad_nan"] == 0 and r["dgrad_rel"] < 4e-3, r
    assert r["wgrad_nan"] == 0 and r["wgrad_rel"] < 2e-4, r      # fp32 output, deterministic split-K


@pytest.mark.parametrize("name", _cases("prologue"))
def test_operand_prologue_and_fused_statistics(name):
    """conv forward / weight gradient reading the producer's RAW output (BatchNorm affine + ReLU applied to the staged
    tiles in shared memory) against cstp_bn_apply followed by the plain kernels: same bf16 operands in the same order, so
    the results -- and the BatchNorm statistics fused into the epilogue -- must be bit-identical."""
    from tools.gpu_kernel_check import run_case
    r = run_case(name)
    assert r["fwd_nan"] == 0 and r["fwd_equal"], r
    assert r.get("stats_equal", True), r
    # (wgrad_gemm with a prologue keeps one M tile per CTA but the plain kernel's split-K factor: same K ranges, same sum order)
    assert r["wgrad_nan"] == 0 and r["wgrad_equal"], r


@pytest.mark.parametrize("name", _cases("linear"))
def test_linear(name):
    from tools.gpu_kernel_check import run_case
    r = run_case(name)
    assert r["nan"] == 0 and r["bf16_rel"] < 4e-3 and r["f32_rel"] < 1e-5, r


def test_elementwise_bn_stem_ema_sgd():
    from tools.gpu_kernel_check import run_case
    r = run_case("elementwise")
    for C in (144, 4096, 83):
        assert r[f"bn{C}_fwd_rel"] < 4e-3 and r[f"bn{C}_dx_rel"] < 4e-3, r
        assert r[f"bn{C}_rm_rel"] < 1e-5 and r[f"bn{C}_rv_rel"] < 1e-5, r
        assert r[f"bn{C}_dgamma_rel"] < 1e-5 and r[f"bn{C}_dbeta_rel"] < 1e-5, r
    assert r["stem_pack_exact"] and r["stem_fwd_padzero"], r
    assert r["stem_fwd_rel"] < 4e-3 and r["stem_wgrad_rel"] < 2e-4, r
    assert r["ema_bitexact"]                                       # r21d_byol.py:331-337: exact fp32 arithmetic
    assert r["sgd_rel"] < 1e-6
    assert abs(r["sgd_norm"][0] - r["sgd_norm"][1]) < 1e-4 * r["sgd_norm"][1]


def test_losses_byol_ce_ntxent():
    from tools.gpu_kernel_check import run_case
    r = run_case("losses")
    assert r["byol_loss_rel"] < 1e-5 and r["byol_grad_rel"] < 1e-5, r
    assert r["ce_loss_rel"] < 1e-5 and r["ce_total_rel"] < 1e-5 and r["ce_grad_rel"] < 1e-5, r
    for rows in (256, 1024, 200):
        assert r[f"ntxent{rows}_loss_rel"] < 1e-5 and r[f"ntxent{rows}_grad_rel"] < 1e-4, r


def test_ragged_and_tiny_geometries():
    """Edge cases: batch 1, odd sizes that leave partial tiles in every tile-space axis, channel counts that are not
    multiples of 16, a single 128-row tile."""
    from tools.gpu_kernel_check import case_conv
    for kw in (dict(N=1, T=3, H=10, W=6, cin=42, cout=85, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1)),
               dict(N=1, T=5, H=6, W=10, cin=85, cout=42, kernel=(3, 1, 1), stride=(2, 1, 1), pad=(1, 0, 0)),
               dict(N=3, T=2, H=14, W=14, cin=170, cout=21, kernel=(1, 3, 3), stride=(1, 2, 2), pad=(0, 1, 1)),
               dict(N=1, T=1, H=2, W=2, cin=16, cout=16, kernel=(1, 1, 1), stride=(1, 1, 1), pad=(0, 0, 0)),
               # 2-D halo layouts (conv fwd / dgrad with a 16-channel tail / wgrad) with partial tiles along h and w
               dict(N=1, T=2, H=40, W=36, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1)),
               dict(N=2, T=1, H=36, W=28, cin=128, cout=240, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1)),
               # slab mode (dgrad of 64 -> 144 1x3x3: four dx rows per tile): rows / columns / frames that do not fill the tiles
               dict(N=3, T=5, H=30, W=36, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1)),
               dict(N=2, T=16, H=28, W=28, cin=64, cout=144, kernel=(1, 3, 3), stride=(1, 1, 1), pad=(0, 1, 1))):
        r = case_conv(**kw)
        assert r["fwd_nan"] == 0 and r["fwd_pad_zero"] and r["fwd_rel"] < 4e-3, (kw, r)
        assert r["dgrad_nan"] == 0 and r["dgrad_rel"] < 4e-3, (kw, r)
        assert r["wgrad_nan"] == 0 and r["wgrad_rel"] < 2e-4, (kw, r)


def test_bn_sync_exchange_protocol_on_one_gpu():
    """csrc/p2p_sync.cu without a second GPU: (a) world 1 is the identity through the slot / flag machinery for many calls;
    (b) two "ranks" with their own buffers on the same device, launched on two streams, exchange rows through the flag
    protocol exactly as two GPUs would (each kernel spins until the other has published)."""
    from cstp_b200 import lib as L
    lib = L.load()
    slots, row_max, n = 4, 64, 48
    err = torch.zeros(1, dtype=torch.int32, device="cuda")

    def buffers(world):
        nbytes = lib.cstp_bn_sync_buffer_bytes(world, slots, row_max)
        bufs = [torch.zeros((nbytes + 3) // 4, dtype=torch.float32, device="cuda") for _ in range(world)]
        return bufs, torch.tensor([b.data_ptr() for b in bufs], dtype=torch.int64, device="cuda")

    bufs, peers = buffers(1)
    for seq in range(1, 11):
        row = torch.randn(n, device="cuda")
        out = torch.empty_like(row)
        L.check(lib.cstp_bn_sync_exchange(row.data_ptr(), n, peers.data_ptr(), 1, 0, slots, row_max, seq, None, out.data_ptr(),
                                          err.data_ptr(), torch.cuda.current_stream().cuda_stream))
        assert torch.equal(out, row)
    bufs, peers = buffers(2)
    s = [torch.cuda.Stream(), torch.cuda.Stream()]
    counters = torch.full((2,), 6, dtype=torch.int32, device="cuda")      # device-side call counters (CUDA-graph form)
    torch.cuda.synchronize()
    for seq in range(1, 13):
        rows = [torch.randn(n, device="cuda"), torch.randn(n, device="cuda")]
        want = rows[0] + rows[1]
        torch.cuda.synchronize()
        for r in (seq % 2, 1 - seq % 2):                     # alternate which "rank" is launched first
            with torch.cuda.stream(s[r]):
                host_seq = seq <= 6          # first half: sequence number from the host, second half: device counter
                L.check(lib.cstp_bn_sync_exchange(rows[r].data_ptr(), n, peers.data_ptr(), 2, r, slots, row_max,
                                                  seq if host_seq else 0,
                                                  None if host_seq else counters[r:r + 1].data_ptr(),
                                                  rows[r].data_ptr(), err.data_ptr(), s[r].cuda_stream))     # in place
        torch.cuda.synchronize()
        assert torch.equal(rows[0], rows[1])                 # same order of summation on both ranks: identical bits
        assert torch.equal(rows[0], want)
    assert int(err.item()) == 0 and counters.tolist() == [12, 12]


def test_batched_weight_pack_equals_the_per_tensor_pack():
    """cstp_pack_weights_batched (one launch for every weight of a network, eight K columns per 16-byte store) writes the
    very bytes of cstp_pack_weight job by job: forward layout, dgrad transpose, stem row-pair layout, ragged channel counts
    (padding rows and columns exactly zero)."""
    from cstp_b200 import ops
    from cstp_b200.ops import pad64
    g = torch.Generator(device="cuda").manual_seed(3)
    jobs, refs = [], []
    for (cout, cin, k, tr) in ((144, 64, (1, 3, 3), 0), (144, 64, (1, 3, 3), 1), (64, 144, (3, 1, 1), 0), (64, 144, (3, 1, 1), 1),
                               (83, 45, (3, 1, 1), 0), (83, 45, (3, 1, 1), 1), (45, 3, (1, 7, 7), 2), (512, 1152, (3, 1, 1), 1),
                               (4096, 512, (), 0), (5, 4096, (), 0)):
        w = torch.randn((cout, cin) + k, device="cuda", generator=g)
        co, ci, taps = ops._pack_dims(w, tr)
        rows, cols = (ci, co) if tr == 1 else (co, ci)
        Rp = (rows + 15) // 16 * 16
        shape = (Rp, taps * pad64(cols))
        a = torch.full(shape, 7.0, device="cuda", dtype=torch.bfloat16)
        b = torch.full(shape, 9.0, device="cuda", dtype=torch.bfloat16)
        ops.pack_weight(w, b, transpose=tr)
        jobs.append((w, a, tr))
        refs.append(b)
    ops.PackList(jobs, "cuda").run()
    torch.cuda.synchronize()
    for (w, a, tr), b in zip(jobs, refs):
        assert torch.equal(a.view(torch.int16), b.view(torch.int16)), (tuple(w.shape), tr)
