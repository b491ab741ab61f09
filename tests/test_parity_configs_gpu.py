"""GPU parity tests at the configurations BASELINE.json names (whole models, full widths), the single-pass TF32
mode over a 20-step rollout, the dlwpbench loop, CUDA-graph replay, and a tensor on a non-current device.

Oracle: oracle/spectral_oracle.py in float64 on the CPU.  Tolerances are written at each assert:
fp32 path (3xTF32 split / exact FFMA) rel-L2 <= 1e-5 (weight gradients that reduce over > 1e5 pixels: 2e-5);
single-pass TF32 mode: 1e-2 over a 20-step rollout (north_star's bound), 3e-3 per step.
"""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

import dlwp_benchmark_b200 as pkg
from dlwp_benchmark_b200 import _lib
from oracle import spectral_oracle as so
from conftest import rel_l2, ROOT

pytestmark = pytest.mark.gpu
DEV = "cuda"
TOL = 1e-5

sys.path.insert(0, ROOT)
import bench  # noqa: E402  (WORKLOADS / build_model: the benchmarked configuration itself)


def _rand(*s, seed=0):
    return torch.randn(*s, generator=torch.Generator().manual_seed(seed))


def _oracle_step(sd, x, y, n_modes, L):
    leaves = {k: v.detach().double().clone().requires_grad_(True) for k, v in sd.items()}
    out = so.fno_forward(leaves, x.double(), n_modes, L)
    loss = F.mse_loss(out, y.double())
    loss.backward()
    return out.detach(), loss.item(), {k: v.grad for k, v in leaves.items()}


def _check_grads(model, ref_grads, tol):
    worst = ("", 0.0)
    for k, p in model.named_parameters():
        assert p.grad is not None, k
        e = rel_l2(p.grad, ref_grads[k])
        if e > worst[1]:
            worst = (k, e)
        assert e < tol, (k, e)
    return worst


def test_cfg2_full_tfno_model_fwd_loss_all_grads_and_graph_replay():
    """The configuration bench.py measures (BASELINE configs[1]): TFNO2D rank 0.8, 64x64, width 64, 16 modes,
    256-wide lifting / projection, batch 64 -> lift_gen + fused head + grouped Tucker paths.  Output, loss and every
    gradient vs the fp64 oracle; then the same step as a captured CUDA graph (what bench.py replays)."""
    wl = bench.WORKLOADS["cfg2"]
    m = bench.build_model(wl)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    B = wl["batch"]
    x, y = _rand(B, 1, 64, 64, seed=21), _rand(B, 1, 64, 64, seed=22)
    yo, lo, go = _oracle_step(sd, x, y, wl["n_modes"], wl["L"])
    m = m.to(DEV)
    xd, yd = x.to(DEV), y.to(DEV)
    out = m(xd)
    loss = F.mse_loss(out, yd)
    loss.backward()
    assert rel_l2(out, yo) < TOL
    assert abs(loss.item() - lo) / abs(lo) < TOL
    _check_grads(m, go, 2e-5)
    eager = {k: p.grad.clone() for k, p in m.named_parameters()}
    del out, loss          # drop the eager autograd graph: its AccumulateGrad nodes belong to the default stream
    # --- captured graph: fwd + MSE + bwd, replayed twice
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            m.zero_grad(set_to_none=True)
            F.mse_loss(m(xd), yd).backward()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    m.zero_grad(set_to_none=True)
    g = torch.cuda.CUDAGraph()
    lbuf = torch.zeros((), device=DEV)
    with torch.cuda.graph(g):
        lg = F.mse_loss(m(xd), yd)
        lg.backward()
        lbuf.copy_(lg.detach())
    for _ in range(2):
        g.replay()
    torch.cuda.synchronize()
    assert abs(lbuf.item() - lo) / abs(lo) < TOL
    for k, p in m.named_parameters():
        assert rel_l2(p.grad, eager[k]) < 1e-6, k          # replay == eager (same kernels, same order)
    _check_grads(m, go, 2e-5)


@pytest.mark.parametrize("workload", ["cfg2", "cfg4"])
def test_bench_dump_outputs_hold_the_last_captured_step(tmp_path, workload):
    """bench.py --dump-outputs through the replayed CUDA graph (FNO arm cfg2, AFNO arm cfg4): the dumped output and
    loss belong to the same step (MSE of the output against the seeded target == the loss; for cfg2 also == the loss
    the step read back), every parameter and gradient is there in float32, and a second run dumps the same arrays."""
    import json
    import subprocess
    import numpy as np
    wl = bench.WORKLOADS[workload]
    runs = []
    for k in range(2):
        d = tmp_path / str(k)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", workload, "--steps", "2",
                            "--warmup", "3", "--skip-cpu", "--skip-roofline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == 2 and (line.get("run") or line["config"])["cuda_graph"]
        runs.append({f[:-4]: np.load(d / f) for f in os.listdir(d)})
    got = runs[0]
    g = torch.Generator().manual_seed(1234)
    if workload == "cfg2":
        m = bench.build_model(wl)
        torch.randn(wl["batch"], 1, wl["H"], wl["W"], generator=g)                            # x
        target = torch.randn(wl["batch"], 1, wl["H"], wl["W"], generator=g)
        assert float(got["loss"]) == line["e2e"]["last_loss"]
    else:
        m = bench._build_afnonet(pkg, wl)
        B, H, W = wl["batch"], wl["H"], wl["W"]
        torch.randn(B, 1, 4, H, W, generator=g), torch.randn(B, 2, 1, H, W, generator=g)      # constants, prescribed
        target = torch.randn(B, 2, wl["cout"], H, W, generator=g)[:, 1:]
    assert got["output"].shape == tuple(target.shape)
    loss = F.mse_loss(torch.from_numpy(got["output"]).double(), target.double()).item()
    assert abs(loss - float(got["loss"])) / float(got["loss"]) < 1e-5
    names = {k for k, _ in m.named_parameters()}
    assert {k[6:] for k in got if k.startswith("param.")} == names
    unused = {"norm.weight", "norm.bias"} if workload == "cfg4" else set()       # AFNONet's final norm: no gradient
    assert {k[5:] for k in got if k.startswith("grad.")} == names - unused
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in got.values())
    assert set(runs[1]) == set(got)
    for k, a in got.items():
        assert np.linalg.norm(runs[1][k] - a) <= 1e-6 * np.linalg.norm(a), k


def test_dlwpbench_shape_whole_model_13_to_8_channels_32x64():
    """dlwpbench FNO (src/dlwpbench/configs/model/fno.yaml: 4 + 9*1 = 13 in, 8 out, 32x64 grid, 12 modes,
    width 32, lifting / projection 256): no fused head (n_out != 1), small-M lifting path."""
    torch.manual_seed(3)
    for cls, rank in ((pkg.FNO, 1.0), (pkg.TFNO, 0.8)):
        m = cls(n_modes=(12, 12), hidden_channels=32, in_channels=13, out_channels=8, lifting_channels=256,
                projection_channels=256, n_layers=4, rank=rank)
        sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
        x, y = _rand(3, 13, 32, 64, seed=31), _rand(3, 8, 32, 64, seed=32)
        yo, lo, go = _oracle_step(sd, x, y, (12, 12), 4)
        m = m.to(DEV)
        xd = x.to(DEV).requires_grad_(True)
        out = m(xd)
        loss = F.mse_loss(out, y.to(DEV))
        loss.backward()
        assert rel_l2(out, yo) < TOL
        assert abs(loss.item() - lo) / abs(lo) < TOL
        _check_grads(m, go, 2e-5)


@pytest.mark.parametrize("name,B", [("cfg3", 1), ("cfg5", 2)])
def test_cfg3_cfg5_full_width_models(name, B):
    """BASELINE configs[2] (256x256) and configs[4] (128x128) at their full width (64 channels, 32 modes, 256-wide
    lifting / projection) with a small batch: output + every gradient (cfg3), forward under no_grad (cfg5)."""
    wl = bench.WORKLOADS[name]
    m = bench.build_model(wl)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    H, W = wl["H"], wl["W"]
    x, y = _rand(B, 1, H, W, seed=41), _rand(B, 1, H, W, seed=42)
    m = m.to(DEV)
    if name == "cfg5":
        with torch.no_grad():
            yo = so.fno_forward({k: v.double() for k, v in sd.items()}, x.double(), wl["n_modes"], wl["L"])
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            out = m(x.to(DEV))
            peak = torch.cuda.max_memory_allocated() - base
        assert rel_l2(out, yo) < TOL
        # under no_grad no pre-activation z is written: the peak is a few [B,64,H,W] activations, not 1 + 2 per layer
        act = B * 64 * H * W * 4
        assert peak < 4.5 * act, (peak, act)
        return
    yo, lo, go = _oracle_step(sd, x, y, wl["n_modes"], wl["L"])
    out = m(x.to(DEV))
    loss = F.mse_loss(out, y.to(DEV))
    loss.backward()
    assert rel_l2(out, yo) < TOL
    assert abs(loss.item() - lo) / abs(lo) < TOL
    _check_grads(m, go, 2e-5)


def test_tf32_single_pass_mode_20_step_rollout_and_train_step():
    """north_star: the TF32 tensor-core path within a stated bound (about 1e-2) over a 20-step rollout.
    sb200_set_tc_mode(1): single-pass kind::tf32 in every tcgen05 kernel.  Bounds: <= 1e-2 after 20 closed-loop
    steps, <= 3e-3 for one forward, <= 1e-2 for the gradients of one train step."""
    lib = _lib.load()
    torch.manual_seed(5)
    m = pkg.FNO(n_modes=(16, 16), hidden_channels=64, in_channels=1, out_channels=1, lifting_channels=256,
                projection_channels=256, n_layers=4)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    x0 = _rand(2, 1, 64, 64, seed=51)
    ref = so.rollout({k: v.double() for k, v in sd.items()}, x0.double(), (16, 16), 4, 20)
    y = _rand(2, 1, 64, 64, seed=52)
    yo, lo, go = _oracle_step(sd, x0, y, (16, 16), 4)
    m = m.to(DEV)
    old = _lib.tc_mode()
    try:
        _lib.set_tc_mode(1)
        outs, x = [], x0.to(DEV)
        with torch.no_grad():
            for _ in range(20):
                x = m(x)
                outs.append(x)
        got = torch.stack(outs, dim=1)
        e1, e20, eall = rel_l2(got[:, 0], ref[:, 0]), rel_l2(got[:, -1], ref[:, -1]), rel_l2(got, ref)
        out = m(x0.to(DEV))
        F.mse_loss(out, y.to(DEV)).backward()
        worst = _check_grads(m, go, 1e-2)
    finally:
        _lib.set_tc_mode(old)
    print(f"tf32 single pass: step-1 {e1:.2e}, step-20 {e20:.2e}, all {eall:.2e}, worst grad {worst}")
    assert e1 < 3e-3 and e20 < 1e-2 and eall < 1e-2
    assert e1 > 1e-6, "mode 1 produced fp32-exact results: the single-pass TF32 path did not run"


@pytest.mark.parametrize("T,ctx", [(5, 1), (57, 1), (6, 2)])
def test_dlwpbench_rollout_loop(T, ctx):
    """FNO2DModule.forward semantics (src/dlwpbench/models/fno/fno.py:64-106): sequence_length 5 (training
    default) and 57 (test default) at context 1, plus a context-2 window; differentiable loop and graph engine."""
    torch.manual_seed(9)
    Cc, Cp, Cg, H, W, B = 4, 1, 8, 32, 64, 2
    m = pkg.FNO(n_modes=(12, 12), hidden_channels=16, in_channels=Cc + (Cp + Cg) * ctx, out_channels=Cg,
                lifting_channels=32, projection_channels=32, n_layers=4)
    sd = {k: v.detach().double() for k, v in m.state_dict().items()}
    c, p, g = _rand(B, 1, Cc, H, W, seed=61), _rand(B, T, Cp, H, W, seed=62), _rand(B, T, Cg, H, W, seed=63) * 0.5
    with torch.no_grad():
        ref = so.dlwp_rollout(sd, c.double(), p.double(), g.double(), ctx, (12, 12), 4)
    m = m.to(DEV)
    cd, pd, gd = c.to(DEV), p.to(DEV), g.to(DEV)
    eng = pkg.DLWPRollout(m, ctx, graph=True)
    got = eng(cd, pd, gd)
    assert got.shape == ref.shape == (B, T - ctx, Cg, H, W)
    tol = TOL if T <= 6 else 5e-5                   # 56 closed-loop steps accumulate rounding
    assert rel_l2(got, ref) < tol
    assert torch.equal(got, eng(cd, pd, gd))        # replay is deterministic
    if T <= 6:
        seq = pkg.dlwp_sequence_forward(m, cd, pd, gd, ctx)
        assert rel_l2(seq, ref) < TOL
        seq.square().mean().backward()                # the loop stays differentiable (BPTT through the window)
        assert all(p_.grad is not None and torch.isfinite(p_.grad).all() for p_ in m.parameters())


def test_standalone_mlp_and_spectralconv_bias_grad_use_the_c_abi():
    """MLP.forward (no torch.matmul) and the bias gradient of a skip-less SpectralConv (sb200_channel_sum)."""
    torch.manual_seed(2)
    lib = _lib.load()
    mlp = pkg.MLP(8, 4, hidden_channels=32, n_layers=2).to(DEV)
    x = _rand(2, 8, 16, 16, seed=71)
    n0 = lib.sb200_kernel_launches()
    xd = x.to(DEV).requires_grad_(True)
    out = mlp(xd)
    out.square().sum().backward()
    assert lib.sb200_kernel_launches() > n0
    xo = x.double().requires_grad_(True)
    w = [p.detach().double().cpu().requires_grad_(True) for p in mlp.parameters()]
    ho = F.conv2d(F.gelu(F.conv2d(xo, w[0], w[1])), w[2], w[3])
    ho.square().sum().backward()
    assert rel_l2(out, ho) < TOL and rel_l2(xd.grad, xo.grad) < TOL
    for p, q in zip(mlp.parameters(), w):
        assert rel_l2(p.grad, q.grad) < TOL
    conv = pkg.SpectralConv(4, 4, (6, 6), fft_norm="forward").to(DEV)
    x = _rand(2, 4, 16, 16, seed=72)
    y = conv(x.to(DEV))
    y.sum().backward()
    assert rel_l2(conv.bias.grad.reshape(-1), torch.full((4,), 2.0 * 16 * 16)) < 1e-6


def test_width_not_multiple_of_4_and_odd_height_fail_loudly():
    m = pkg.FNO(n_modes=(4, 4), hidden_channels=8, in_channels=1, out_channels=1, lifting_channels=16,
                projection_channels=16, n_layers=2).to(DEV)
    for shape in ((1, 1, 16, 18), (1, 1, 15, 16)):
        with pytest.raises(_lib.SpectralB200Error):
            m(torch.randn(*shape, device=DEV))


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_tensor_on_non_current_device():
    """ADVICE r1: kernels must launch on the stream / device of the tensor, not of the current device."""
    torch.manual_seed(4)
    m = pkg.FNO(n_modes=(12, 12), hidden_channels=32, in_channels=1, out_channels=1, lifting_channels=256,
                projection_channels=256, n_layers=2)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    x, y = _rand(2, 1, 64, 64, seed=81), _rand(2, 1, 64, 64, seed=82)
    yo, lo, go = _oracle_step(sd, x, y, (12, 12), 2)
    assert torch.cuda.current_device() == 0
    m = m.to("cuda:1")
    out = m(x.to("cuda:1"))
    F.mse_loss(out, y.to("cuda:1")).backward()
    torch.cuda.synchronize(1)
    assert out.device.index == 1 and torch.cuda.current_device() == 0
    assert rel_l2(out, yo) < TOL
    _check_grads(m, go, 2e-5)
    a = pkg.AFNO2D(32, num_blocks=4).to("cuda:1")
    z = a(torch.randn(1, 8, 16, 32, device="cuda:1"))
    z.sum().backward()
    assert z.device.index == 1 and torch.isfinite(z).all()
