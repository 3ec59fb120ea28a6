"""bench.py pieces that run without a GPU: the reference arm's JSON line (the CPU oracle port on a bounded sample), the
helper behind roofline.traffic and the --dump-outputs writer; on a GPU, --dump-outputs through the native arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line_has_the_contract_keys_and_names_its_sample():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1                      # ONE JSON line
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "clips/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"] == "clips/sec, r21d_byol pretrain step, 16x112x112"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "clips/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the arm runs a bounded sample of the batch-60 workload and says so in its config
    assert d["config"]["per_gpu_batch"] == 60 and d["config"]["sampled_batch"] == 2 and d["config"]["same_config"] is False


def test_roofline_traffic_comes_from_a_committed_capture_with_its_provenance():
    sys.path.insert(0, ROOT)
    import bench
    per_launch, src = bench.ncu_traffic("conv_halo_kernel", 60)
    assert src.startswith("profiles/r02_ncu_conv_halo_b60_dram.csv") and "commit" in src
    assert 1.5e9 < per_launch < 2.5e9          # ~1.88 GB per launch = the algorithmic bytes of the layers it runs
    assert bench.ncu_traffic("conv_halo_kernel", 7) == (None, None)


def test_dump_outputs_writes_the_loss_vector_and_a_fixed_sample_of_the_state(tmp_path):
    """--dump-outputs: float32 / float64 arrays, within 64 MB for the flagship model, the same positions on every run."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from cstp_b200.models.pace.r21d_byol import R21DBYOL
    torch.manual_seed(1)
    state = R21DBYOL(pretrain=True).state_dict()
    losses = torch.arange(8, dtype=torch.float32)
    total = bench.dump_outputs(str(tmp_path / "a"), losses, state)
    assert total <= bench.DUMP_LIMIT
    assert bench.dump_outputs(str(tmp_path / "b"), losses, state) == total
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(["losses.npy"] + [f"state.{k}.npy" for k in state])
    assert sum((tmp_path / "a" / n).stat().st_size for n in names) < bench.DUMP_LIMIT
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b), n
    assert np.array_equal(np.load(tmp_path / "a" / "losses.npy"), losses.numpy())
    w = state["online_net.conv2.block1.conv1.spatial_conv.weight"].reshape(-1)
    got = np.load(tmp_path / "a" / "state.online_net.conv2.block1.conv1.spatial_conv.weight.npy")
    assert w.numel() > bench.DUMP_SAMPLE and got.shape == (bench.DUMP_SAMPLE,) and np.isin(got, w.numpy()).all()
    bn = state["online_net.conv1.bn.running_mean"]
    assert np.array_equal(np.load(tmp_path / "a" / "state.online_net.conv1.bn.running_mean.npy"), bn.numpy())
    assert np.load(tmp_path / "a" / "state.online_net.conv1.bn.num_batches_tracked.npy").dtype == np.float64


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_repeat_run_to_run(tmp_path):
    """--dump-outputs through main() on the GPU: the loss vector of the last timed step (the one the JSON line reports) and
    the CUDA-resident model state it left, bit-identical on two runs with the same arguments."""
    import numpy as np

    def run(d):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "3",
                              "--no-cpu-baseline", "--dump-outputs", str(d)], capture_output=True, text=True, timeout=900,
                             cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
        return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])

    line = run(tmp_path / "a")
    run(tmp_path / "b")
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(p.name for p in (tmp_path / "b").iterdir()) and len(names) == 352
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert np.isfinite(a).all() and np.array_equal(a, b), n
    losses = np.load(tmp_path / "a" / "losses.npy")
    assert losses.tolist() == [*line["losses_last_step"]["ce"], losses[6], line["losses_last_step"]["byol"]]


def test_bench_rejects_a_run_without_timed_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert out.returncode != 0 and "--steps must be at least 1" in out.stderr


def test_watchdog_prints_the_measured_line_when_a_sub_record_hangs():
    """bench.py at N > 1: a config-5 sub-record that never returns (a lost peer) must not lose the batch-60 line."""
    code = ("import sys, time; sys.path.insert(0, %r); import bench\n"
            "line = {'metric': 'm', 'value': 1.0}\n"
            "bench.run_with_watchdog(0.3, lambda: time.sleep(30), lambda: bench.bail_out(line, 'config5', 'too slow'))\n"
            "print('not reached')\n") % ROOT
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=60)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0]) == {"metric": "m", "value": 1.0, "config5": {"error": "too slow"}}
    # and a sub-record that returns in time passes its result through, the timer cancelled
    sys.path.insert(0, ROOT)
    import bench
    assert bench.run_with_watchdog(5.0, lambda: {"ok": 1}, lambda: (_ for _ in ()).throw(AssertionError("fired"))) == {"ok": 1}
