#!/usr/bin/env python
"""Headline benchmark: FNO-family train step (fwd + MSE + bwd + Adam) samples/s on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg2|cfg1|cfg3]
                    [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, NCCL); rank 0 prints ONE JSON line.
--dump-outputs DIR: after the timed steps, rank 0 writes what the last step handed its caller as DIR/<name>.npy (see
dump_outputs); inputs and weights are seeded, so two builds of the project can be compared output for output.

Workload at N=1 (BASELINE.json configs[1], the config the metric's target is quoted on):
TFNO2D (Tucker rank 0.8) on 64x64 synthetic fields, 1 -> 1 channels, width 64, 16 modes, 4 layers,
lifting/projection 256, batch 64 PER GPU (weak scaling), fp32.

Keys beyond the base contract:
  roofline      dominant kernel (by device time) of the spectral path, timed alone with CUDA events
                on the launching stream; algorithmic bytes per launch are stated in DESIGN.md
  cpu_baseline  the oracle (torch CPU restatement of the reference path) on this box's host cores,
                on a bounded sample (smaller batch) of the same workload
  e2e           same metric through the public nn.Module API with pinned-host inputs copied H2D and
                the loss read back D2H inside the timed region every step
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: dict(model kwargs, grid, per-gpu batch, tucker)
    "cfg1": dict(desc="FNO2D 64x64 in1 width32 modes12 L4 batch8 (BASELINE configs[0], CPU-runnable)",
                 n_modes=(12, 12), hidden=32, cin=1, cout=1, L=4, lift=256, proj=256, H=64, W=64, batch=8, rank=0.0),
    "cfg2": dict(desc="TFNO2D(Tucker rank 0.8) 64x64 in1 width64 modes16 L4 batch64/GPU (BASELINE configs[1])",
                 n_modes=(16, 16), hidden=64, cin=1, cout=1, L=4, lift=256, proj=256, H=64, W=64, batch=64, rank=0.8),
    "cfg2d": dict(desc="FNO2D(dense) 64x64 in1 width64 modes16 L4 batch64/GPU",
                  n_modes=(16, 16), hidden=64, cin=1, cout=1, L=4, lift=256, proj=256, H=64, W=64, batch=64, rank=0.0),
    "cfg3": dict(desc="FNO2D 256x256 in1 width64 modes32 L4 batch64/GPU (BASELINE configs[2])",
                 n_modes=(32, 32), hidden=64, cin=1, cout=1, L=4, lift=256, proj=256, H=256, W=256, batch=64, rank=0.0),
    # the two below are not train-step lines of the FNO metric: they have their own metric names
    "cfg4": dict(desc="FourCastNet AFNONet (dlwpbench flavour): 32x64 grid, patch 1x1, 4 const + 1 prescribed + 8 prognostic = 13 in / "
                      "8 out channels, embed 256, depth 8, num_blocks 8, mlp_ratio 4, pos_embed, batch 16/GPU, single step "
                      "(BASELINE configs[3])",
                 kind="afnonet", embed=256, nb=8, depth=8, H=32, W=64, batch=16, cin=13, cout=8),
    "cfg4f": dict(desc="AFNO2D filter stack only: 8 x AFNO2D(embed 256, 8 blocks) on 32x64 tokens, batch 16/GPU",
                  kind="afno", embed=256, nb=8, depth=8, H=32, W=64, batch=16),
    "cfg5": dict(desc="FNO2D closed-loop rollout 128x128 in1 width64 modes32 L4, 512 initial conditions/GPU x 100 steps "
                      "(BASELINE configs[4])",
                 kind="rollout", n_modes=(32, 32), hidden=64, cin=1, cout=1, L=4, lift=256, proj=256, H=128, W=128,
                 batch=512, rank=0.0, rollout_steps=100),
}


def log(msg):
    sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


DUMP_BYTES = 64_000_000


def dump_outputs(path, arrays, limit=DUMP_BYTES):
    """Write ``arrays`` (name -> tensor; None entries are skipped) as ``path/<name>.npy`` in float32 (float64 stays
    float64), at most ``limit`` bytes of files in all.  Arrays are taken smallest first and each is written whole when
    it fits an equal share of what is left.  One that does not is written as a flat 1-D sample: its elements at the
    distinct flat indices among that many draws from a fixed seed (with replacement, so somewhat fewer than the share),
    in index order, so the same workload gives the same sample on every run; neither the shape nor the indices are
    written."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    items = sorted(((k, v) for k, v in arrays.items() if v is not None), key=lambda kv: kv[1].numel())
    left = limit
    for i, (name, t) in enumerate(items):
        t = t.detach()
        t = t if t.dtype == torch.float64 else t.float()
        share = left // (len(items) - i) - 128                     # 128: the .npy header
        if t.numel() * t.element_size() > share:
            idx = torch.randint(t.numel(), (max(share, 0) // t.element_size(),), generator=torch.Generator().manual_seed(0))
            t = t.reshape(-1)[idx.unique().to(t.device)]            # sorted, distinct
        fn = os.path.join(path, name + ".npy")
        np.save(fn, t.cpu().numpy())
        left -= os.path.getsize(fn)


def _train_step_outputs(out, loss, model):
    """What one train step hands its caller: the model output, the loss, every gradient and every updated parameter."""
    d = {"output": out, "loss": loss}
    for k, p in model.named_parameters():
        d["param." + k] = p
        d["grad." + k] = p.grad
    return d


def build_model(wl, seed=1234):
    import torch
    import dlwp_benchmark_b200 as pkg
    torch.manual_seed(seed)
    cls = pkg.TFNO if wl["rank"] > 0 else pkg.FNO
    return cls(n_modes=wl["n_modes"], hidden_channels=wl["hidden"], in_channels=wl["cin"], out_channels=wl["cout"],
               lifting_channels=wl["lift"], projection_channels=wl["proj"], n_layers=wl["L"],
               rank=wl["rank"] if wl["rank"] > 0 else 1.0)


# ----------------------------------------------------------------------------------------
# clocks sampling (recipe in B200_PROFILING.md)
# ----------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.samples, self.stop = index, [], threading.Event()
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.samples.append([s.strip() for s in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0])); mx = max(mx, float(s[1]))
                for n, v in zip(names, s[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ----------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle on host cores, bounded sample
# ----------------------------------------------------------------------------------------
def _oracle_step_fn(wl, sample_batch, device):
    """One train step (fwd + MSE + bwd + Adam) of the oracle restatement of the reference path -- plain
    torch.fft / einsum / conv2d, fp32 -- on ``device``.  Returns (step, sync)."""
    import torch
    from oracle import spectral_oracle as so
    m = build_model(wl)
    sd = {k: v.detach().clone().to(device).requires_grad_(True) for k, v in m.state_dict().items()}
    opt = torch.optim.Adam(list(sd.values()), lr=1e-3, **({"capturable": True} if device != "cpu" else {}))
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(sample_batch, wl["cin"], wl["H"], wl["W"], generator=g).to(device)
    y = torch.randn(sample_batch, wl["cout"], wl["H"], wl["W"], generator=g).to(device)

    def step():
        opt.zero_grad(set_to_none=True)
        out = so.fno_forward(sd, x, wl["n_modes"], wl["L"])
        loss = torch.nn.functional.mse_loss(out, y)
        loss.backward()
        opt.step()
        return loss
    return step


def cpu_oracle_rate(wl, sample_batch, steps, warmup):
    """fwd + MSE + bwd + Adam of the oracle restatement (torch CPU, fp32, all host threads); total time / steps."""
    import torch
    torch.set_num_threads(os.cpu_count() or 1)
    step = _oracle_step_fn(wl, sample_batch, "cpu")
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    per = (time.perf_counter() - t0) / steps
    return sample_batch / per, per, torch.get_num_threads()


def gpu_torch_rate(wl, batch, steps=10, warmup=3):
    """COMPARISON ONLY (north_star: "cuFFT and torch.fft on the GPU are reported only as comparisons"): the same
    oracle module -- torch.fft (cuFFT) + einsum + conv2d, fp32, TF32 off -- on this B200, eager and as a CUDA graph.
    Nothing of this is on the product path."""
    import torch
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    out = {"what": "oracle restatement of the reference path (torch.fft/cuFFT + einsum + conv2d, fp32, allow_tf32=False) "
                   "on the same GPU, fwd+MSE+bwd+Adam", "batch": batch}
    try:
        step = _oracle_step_fn(wl, batch, "cuda")

        def timed(fn):
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) * 1e-3 / steps
        t = timed(step)
        out["eager"] = {"ms_per_step": t * 1e3, "samples_per_s": batch / t}
        try:
            s = torch.cuda.Stream()
            s.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(s):
                step()
            torch.cuda.current_stream().wait_stream(s)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                step()
            t = timed(g.replay)
            out["cuda_graph"] = {"ms_per_step": t * 1e3, "samples_per_s": batch / t}
            del g
        except Exception as ex:  # noqa: BLE001
            out["cuda_graph"] = {"error": repr(ex)[:200]}
            torch.cuda.synchronize()
    except Exception as ex:  # noqa: BLE001
        out["error"] = repr(ex)[:200]
    return out


def cpu_rollout_rate(wl, n_ics=2, n_steps=3):
    """cfg5 on the host cores: closed-loop rollout of the oracle FNO on a bounded sample (a few ICs x a few steps)."""
    import torch
    from oracle import spectral_oracle as so
    torch.set_num_threads(os.cpu_count() or 1)
    m = build_model(wl)
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    x0 = torch.randn(n_ics, wl["cin"], wl["H"], wl["W"], generator=torch.Generator().manual_seed(1234))
    with torch.no_grad():
        so.rollout(sd, x0, wl["n_modes"], wl["L"], 1)
        t0 = time.perf_counter()
        so.rollout(sd, x0, wl["n_modes"], wl["L"], n_steps)
        dt = time.perf_counter() - t0
    return {"value": n_ics * n_steps / dt, "unit": "IC-steps/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{n_ics} initial conditions x {n_steps} closed-loop steps of the oracle FNO ({dt:.1f} s of CPU work)"}


def cpu_afno_rate(wl, steps=3):
    """cfg4 on the host cores: fwd + MSE + bwd of a stack of AFNO2D filters, oracle/afno_oracle.py (pinned against the
    reference class by tests/golden/afno2d_*.npz), full per-GPU batch."""
    import torch
    from oracle import afno_oracle as ao
    torch.set_num_threads(os.cpu_count() or 1)
    g = torch.Generator().manual_seed(1234)
    C, nb, bs = wl["embed"], wl["nb"], wl["embed"] // wl["nb"]
    ps = [[(0.02 * torch.randn(*s, generator=g)).requires_grad_(True)
           for s in ((2, nb, bs, bs), (2, nb, bs), (2, nb, bs, bs), (2, nb, bs))] for _ in range(wl["depth"])]
    x = torch.randn(wl["batch"], wl["H"], wl["W"], C, generator=g)
    y = torch.randn(wl["batch"], wl["H"], wl["W"], C, generator=g)

    def step():
        h = x
        for w1, b1, w2, b2 in ps:
            h = ao.afno2d_fft(h, w1, b1, w2, b2, nb)
        torch.nn.functional.mse_loss(h, y).backward()
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": wl["batch"] / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"batch {wl['batch']}, {wl['depth']} AFNO2D filters fwd+MSE+bwd, {steps} steps after 1 warm-up "
                      f"({(steps + 1) * dt:.1f} s of CPU work), oracle pinned to the reference class"}


def _config(wl, world):
    """The ``config`` object both arms print (identical keys and values: the driver compares them)."""
    return {"workload": wl["desc"], "global_batch": wl["batch"] * world, "grid": [wl["H"], wl["W"]],
            "parallelism": f"dp{world}", "step": "fwd+MSE+bwd+Adam" + ("+allreduce" if world > 1 else ""),
            "l2": "per-step working set (activations of 4 layers + 256-ch lifting/projection, >1 GB) exceeds the 126 MB L2"}


def _cpu_sample(wl):
    """Samples per CPU step: the full per-GPU batch on the 64x64 grids (about 10 s of CPU work for the whole
    measurement on the GPU box's host cores), a bounded slice of it on the large grids."""
    if wl["H"] * wl["W"] <= 64 * 64:
        return wl["batch"]
    return max(1, min(wl["batch"], 4 if wl["H"] * wl["W"] <= 128 * 128 else 2))


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    sample = _cpu_sample(wl)
    steps, warmup = args.steps, args.warmup
    rate, med, cores = cpu_oracle_rate(wl, sample, steps, warmup)
    line = {
        "impl": "reference", "metric": "FNO2D train samples/s (fwd+bwd)", "value": rate, "unit": "samples/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": med * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config(wl, world),
        "note": "reference path = oracle restatement of neuralop@05c01c3 (not vendored by the reference, not "
                "installable here: parity unpinned) on the box's host cores; rank 0 only, one GPU's batch per step",
        "cpu_baseline": {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
                         "sample": f"batch {sample} of {wl['batch']} per step, fwd+MSE+bwd+Adam, {steps} steps after "
                                   f"{warmup} warm-up"},
        "e2e": {"value": rate, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------
# per-kernel roofline of the spectral path (timed alone, CUDA events on the launching stream)
# ----------------------------------------------------------------------------------------
def kernel_rooflines(wl, peak_gbs, reps=10):
    import torch
    from dlwp_benchmark_b200 import ops
    from dlwp_benchmark_b200.plan import fno_plan
    dev = torch.device("cuda")
    B, C, H, W = wl["batch"], wl["hidden"], wl["H"], wl["W"]
    half = [wl["n_modes"][0], wl["n_modes"][1] // 2 + 1]
    plan = fno_plan(dev, H, W, half)
    My, Mx = plan.My, plan.Mx
    M = My * Mx
    P = B * C * H * W
    x = torch.randn(B, C, H, W, device=dev)
    g = torch.randn(B, C, H, W, device=dev)
    z = torch.randn(B, C, H, W, device=dev)
    Wc = torch.randn(C, C, My, Mx, 2, device=dev) * 0.1
    ws = torch.randn(C, C, device=dev) * 0.1
    bv = torch.randn(C, device=dev)
    Xh = ops.analysis(plan, 0, x)
    Yh = ops.mix_fwd(Xh, Wc)
    Phi = ops.coldft_inv(plan, 0, Yh)
    flush = torch.empty(192 * 1024 * 1024 // 4, device=dev)     # > 126 MB L2
    spec = 8 * B * C * M                                         # bytes of one [B,C,My,Mx] complex tensor
    tb = 8 * B * C * H * Mx                                      # bytes of T / Phi
    cases = {
        "analysis": (lambda: ops.analysis(plan, 0, x), 4 * P + spec),
        "modes_gemm(mix_fwd)": (lambda: ops.mix_fwd(Xh, Wc), 2 * spec + 8 * C * C * M),
        "modes_gemm(wgrad)": (lambda: ops.mix_bwd_weight(Xh, Yh), 2 * spec + 8 * C * C * M),
        "coldft_inv": (lambda: ops.coldft_inv(plan, 0, Yh), spec + tb),
        "rowidft_pointwise(fwd)": (lambda: ops.rowidft_pointwise(plan, 0, Phi, x, ws, C, 1, bv, None, B, C, C, 0, True,
                                                                 want_z=True), tb + 4 * P + 8 * P),
        "rowidft_pointwise(bwd)": (lambda: ops.rowidft_pointwise(plan, 1, Phi, g, ws, 1, C, None, z, B, C, C, 1, False),
                                   tb + 8 * P + 4 * P),
        "pointwise_wgrad": (lambda: ops.pointwise_wgrad(g, x), 8 * P),
    }
    # lifting (1 -> 256 -> C) and projection (C -> 256 -> 1) MLPs: SURVEY row f1, 256-channel hidden tensor on chip
    LP = wl["lift"]
    if wl["cin"] == 1 and wl["cout"] == 1 and LP == 256 and ops.lift_supported(C, LP, H * W) \
            and ops.mlp_head_supported(C, LP, 1, H * W):
        x1 = torch.randn(B, 1, H, W, device=dev)
        g1 = torch.randn(B, 1, H, W, device=dev)
        w1 = torch.randn(LP, device=dev) * 0.5
        b1 = torch.randn(LP, device=dev) * 0.1
        W2 = torch.randn(C, LP, device=dev) * 0.05
        Wh = torch.randn(LP, C, device=dev) * 0.1
        wo = torch.randn(LP, device=dev) * 0.05
        bo = torch.zeros(1, device=dev)
        P1 = B * H * W
        gz1 = ops.mlp_head_bwd(x, Wh, b1, wo, g1)[0]
        cases.update({
            "lift_fwd": (lambda: ops.lift_fwd(x1, w1, b1, W2, bv), 4 * P1 + 4 * P),
            "lift_wgrad": (lambda: ops.lift_wgrad(g, x1, w1, b1), 4 * P + 4 * P1),
            "lift_tail_bwd": (lambda: ops.lift_tail_bwd(g, W2, w1, b1, x1), 4 * P + 4 * P1),
            "mlp_head_fwd": (lambda: ops.mlp_head_fwd(x, Wh, b1, wo, bo), 4 * P + 4 * P1),
            # the three kernels of the projection backward as they stand (gz1 [B,256,H,W] round-trips HBM):
            "mlp_head_bwd(gz1 out)": (lambda: ops.mlp_head_bwd(x, Wh, b1, wo, g1), 4 * P + 4 * P1 + 4 * B * LP * H * W),
            "head_dgrad(256->C)": (lambda: ops.rowidft_pointwise(plan, 1, None, gz1, Wh, 1, C, None, None, B, LP, C, 1,
                                                                 False), 4 * B * LP * H * W + 4 * P),
            "head_wgrad(256xC)": (lambda: ops.pointwise_wgrad(gz1, x, want_bias=False), 4 * B * LP * H * W + 4 * P),
        })
    out = {}
    for name, (fn, nbytes) in cases.items():
        for _ in range(3):
            fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e-3)
        t = sum(ts) / len(ts)
        out[name] = {"ms": t * 1e3, "alg_bytes": nbytes, "achieved_gbs": nbytes / t / 1e9,
                     "frac": nbytes / t / 1e9 / peak_gbs}
    return out


def _finish(world, graphs=()):
    """End of a rank's work: release the CUDA graphs that captured the NCCL communicator FIRST (destroying a
    communicator that a live graph still references is what blocked in round 1), then a barrier and a normal
    ``destroy_process_group()``.  A 45 s watchdog turns a teardown that still hangs into an exit instead of a burnt
    GPU lease (it reports itself on stderr; every result has been printed and flushed by then)."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world <= 1:
        return
    import torch
    import torch.distributed as dist

    def _bail():
        sys.stderr.write("[bench] destroy_process_group did not return within 45 s: leaving through os._exit\n")
        sys.stderr.flush()
        os._exit(0)
    wd = threading.Timer(45.0, _bail)
    wd.daemon = True
    wd.start()
    torch.cuda.synchronize()
    for g in graphs:
        if g is not None:
            g.reset()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    wd.cancel()


def _peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        v = float(json.load(open(peaks_path))["hbm_gbs"])
        if v > 0:
            return v, "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:  # noqa: BLE001  (absent or unreadable file: the recipe's stated fallback)
        pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def _ncu_table_path(rel=False):
    """newest committed per-kernel table of an `ncu --set full` capture of the cfg2 step (profiles/r*_cfg2_ncu_full*.json)"""
    import glob
    c = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_cfg2_ncu_full*.json")))
    p = c[-1] if c else os.path.join(ROOT, "profiles", "r01_cfg2_ncu_full_s5f.json")
    return os.path.relpath(p, ROOT) if rel else p


def _ncu_traffic(kernel_substr, approx_read_bytes=None):
    """dram read+write bytes per launch of a kernel from the committed `ncu --set full` capture of this workload
    (profiles/r01_cfg2_ncu_full_s5f.json); None when the capture has no such kernel."""
    path = _ncu_table_path()
    try:
        table = json.load(open(path))
    except Exception:
        return None
    best = None
    for name, rows in table.items():
        if kernel_substr not in name:
            continue
        for r in rows:
            if best is None or (approx_read_bytes is not None and
                                abs(r["dram_read_bytes"] - approx_read_bytes) < abs(best["dram_read_bytes"] - approx_read_bytes)):
                best = r
    return None if best is None else int(best["dram_read_bytes"] + best["dram_write_bytes"])


def _timed(step, steps, warmup, world, local_rank, dist):
    """W warm-up steps, then K steps bracketed by barrier + synchronize; returns (seconds, clocks)."""
    import torch
    for _ in range(warmup):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as cs:
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e-3, cs.summary()


# ----------------------------------------------------------------------------------------
# cfg4: AFNO2D filter stack (train step), cfg5: closed-loop rollout (inference)
# ----------------------------------------------------------------------------------------
def _tf_peak():
    """dense TF32 tensor peak used for the GEMM-bound stages: half of the measured dense bf16 rate"""
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk.get("bf16_tflops_sustained") or pk["bf16_tflops"]) / 2, "MEASURED_PEAKS.json bf16_tflops_sustained / 2 (kind::tf32 runs at half the bf16 rate)"
    except Exception:  # noqa: BLE001
        return 1100.0 / 2, "fallback: nominal 1.1 PFLOP/s dense tf32 (B200_PROFILING.md) / 2"


def cpu_afnonet_rate(wl, steps=2):
    """cfg4 on the host cores: one train step (fwd + MSE + bwd) of the oracle restatement of the reference AFNONet
    (oracle/afno_oracle.py, pinned to the reference classes by tests/golden/fcn_*.npz), bounded batch."""
    import torch
    from oracle import afno_oracle as ao
    import dlwp_benchmark_b200 as pkg
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(1234)
    net = _build_afnonet(pkg, wl)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in net.state_dict().items()}
    Bs = max(1, min(wl["batch"], 4))
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(Bs, wl["cin"], wl["H"], wl["W"], generator=g)
    y = torch.randn(Bs, wl["cout"], wl["H"], wl["W"], generator=g)

    def step():
        for v in sd.values():
            v.grad = None
        out = ao.afnonet_step(sd, x, (1, 1), wl["depth"], wl["nb"])
        torch.nn.functional.mse_loss(out, y).backward()
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": Bs / dt, "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"batch {Bs} of {wl['batch']}, fwd+MSE+bwd, {steps} steps after 1 warm-up ({(steps + 1) * dt:.1f} s of CPU "
                      "work), oracle restatement pinned to the reference classes"}


def _build_afnonet(pkg, wl):
    return pkg.AFNONet(img_height=wl["H"], img_width=wl["W"], patch_size=(1, 1), constant_channels=4, prescribed_channels=1,
                       prognostic_channels=wl["cout"], embed_dim=wl["embed"], depth=wl["depth"], mlp_ratio=4.,
                       num_blocks=wl["nb"], context_size=1, use_pos_embed=True)


def run_afno(args, wl, rank, world, local_rank):
    """cfg4: train step of the dlwpbench FourCastNet (AFNONet) -- or, for ``cfg4f``, of the bare AFNO2D filter stack."""
    import torch
    import torch.distributed as dist
    import dlwp_benchmark_b200 as pkg
    from dlwp_benchmark_b200 import _lib
    from dlwp_benchmark_b200.ddp import GradSync
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1234)
    full = wl["kind"] == "afnonet"
    B, H, W, C = wl["batch"], wl["H"], wl["W"], wl["embed"]
    g = torch.Generator().manual_seed(1234 + rank)
    # output of the latest step (inside the graph: its static output), detached: holding its autograd graph would carry
    # the parameters' AccumulateGrad nodes of an eager step, bound to the eager stream, into the graph capture
    last = {}
    if full:
        model = _build_afnonet(pkg, wl).to(dev)
        host = [torch.randn(B, 1, 4, H, W, generator=g).pin_memory(), torch.randn(B, 2, 1, H, W, generator=g).pin_memory(),
                torch.randn(B, 2, wl["cout"], H, W, generator=g).pin_memory()]
        dv = [t.to(dev) for t in host]

        def fwd_loss():
            out = model(constants=dv[0], prescribed=dv[1], prognostic=dv[2])      # [B, 1, 8, H, W]
            last["out"] = out.detach()
            return torch.nn.functional.mse_loss(out, dv[2][:, 1:])
    else:
        model = torch.nn.Sequential(*[pkg.AFNO2D(C, num_blocks=wl["nb"]) for _ in range(wl["depth"])]).to(dev)
        host = [torch.randn(B, H, W, C, generator=g).pin_memory(), torch.randn(B, H, W, C, generator=g).pin_memory()]
        dv = [t.to(dev) for t in host]

        def fwd_loss():
            out = model(dv[0])
            last["out"] = out.detach()
            return torch.nn.functional.mse_loss(out, dv[1])
    params = list(model.parameters())
    opt = torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)
    sync = GradSync(params, world) if world > 1 else None
    loss_buf = torch.zeros((), device=dev)
    hloss = torch.zeros((), pin_memory=True)
    lib = _lib.load()
    if args.tc_mode is not None:
        _lib.set_tc_mode(args.tc_mode)

    def step_eager():
        if sync:
            sync.zero()
        else:
            opt.zero_grad(set_to_none=True)
        loss = fwd_loss()
        loss.backward()
        loss_buf.copy_(loss.detach())
        if sync:
            sync.allreduce()
        opt.step()

    step_eager(); torch.cuda.synchronize()
    n0 = lib.sb200_kernel_launches()
    step_eager(); torch.cuda.synchronize()
    launches = int(lib.sb200_kernel_launches() - n0)
    step = step_eager
    graph = None
    if not args.no_graph:
        s = torch.cuda.Stream(); s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                step_eager()
        torch.cuda.current_stream().wait_stream(s); torch.cuda.synchronize()
        if sync is None:
            opt.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            if sync:
                sync.zero()
            loss = fwd_loss()
            loss.backward()
            loss_buf.copy_(loss.detach())
            if sync:
                sync.allreduce()
            opt.step()
        step = graph.replay
    t_dev, clocks = _timed(step, args.steps, args.warmup, world, local_rank, dist)

    def step_e2e():
        for d, hsrc in zip(dv, host):
            d.copy_(hsrc, non_blocking=True)
        step()
        hloss.copy_(loss_buf, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t_e2e, _ = _timed(step_e2e, args.steps, 3, world, local_rank, dist)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, _train_step_outputs(last["out"], loss_buf, model))
    tt = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = tt.tolist()
    if rank == 0:
        peak, peak_src = _peak()
        P = B * H * W * C
        per = t_dev / args.steps
        if full:
            # GEMM-bound: the token MLP (2 Linear layers of C x 4C, fwd + dgrad + wgrad = 3 x 2 GEMMs) dominates the flops;
            # algorithmic flops = fp32 GEMM flops (2MNK), NOT multiplied by the 3 tf32 passes of the parity mode
            T = B * H * W
            mlp = 6 * 2 * T * C * 4 * C
            bs = C // wl["nb"]
            kept = (H // 2 + 1)
            ntok_f = B * min(2 * kept, H) * min(kept, W // 2 + 1)
            afno = 3 * (2 * 8 * ntok_f * wl["nb"] * bs * bs) + 3 * 2 * (4 * P * min(kept, W // 2 + 1) + 8 * B * C * min(kept, W // 2 + 1) * H * min(2 * kept, H))
            flops = wl["depth"] * (mlp + afno) + 3 * 2 * T * C * (wl["cin"] + wl["cout"])
            tpeak, tsrc = _tf_peak()
            roof = {"bound": "tensor", "kernel": "whole AFNONet train step (tcgen05 GEMMs of the token MLP dominate)",
                    "achieved": flops / per / 1e12, "peak": tpeak, "unit": "TFLOP/s", "frac": flops / per / 1e12 / tpeak,
                    "traffic": None, "peak_source": tsrc, "alg_flops": flops,
                    "note": "algorithmic fp32 flops (2MNK per GEMM, fwd+dgrad+wgrad) over the whole-step time (includes Adam, "
                            "LayerNorm, the AFNO2D filters); the fp32-parity mode issues 3 tf32 MMAs per product, so 1/3 of the "
                            "tf32 peak is the ceiling of this mode"}
            metric, cpu = "FourCastNet (AFNONet) train samples/s (fwd+bwd)", None
            if world == 1 and not args.skip_cpu:
                cpu = cpu_afnonet_rate(wl)
        else:
            alg = 20 * P * wl["depth"]        # per layer: fwd 8P (read x, write y) + bwd 12P (read gy, x for the masks/weights, write gx)
            roof = {"bound": "hbm", "kernel": "AFNO2D layer (all kernels of one layer, fwd+bwd)",
                    "achieved": alg / per / 1e9, "peak": peak, "unit": "GB/s", "frac": alg / per / 1e9 / peak, "traffic": None,
                    "peak_source": peak_src, "alg_bytes": alg,
                    "note": "whole-step time over 20*P bytes per layer (includes Adam and the loss)"}
            metric = "AFNO2D filter stack train samples/s (fwd+bwd)"
            cpu = cpu_afno_rate(wl) if (world == 1 and not args.skip_cpu) else None
        line = {"metric": metric, "value": B * world * args.steps / t_dev,
                "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["desc"], "global_batch": B * world, "grid": [H, W], "parallelism": f"dp{world}",
                           "step": "fwd+MSE+bwd+Adam(fused)", "cuda_graph": step is not step_eager,
                           "tc_mode": int(_lib.tc_mode()),
                           "l2": "working set (saved activations of 8 blocks incl. the 4x hidden tensors, > 2 GB) exceeds the 126 MB L2"},
                "clocks": clocks,
                "e2e": {"value": B * world * args.steps / t_e2e, "unit": "samples/s",
                        "h2d_bytes_per_step": sum(t.numel() for t in host) * 4 * world, "d2h_bytes_per_step": 4 * world,
                        "ms_per_step": t_e2e / args.steps * 1e3},
                "gpu_launches": launches * args.steps,
                "roofline": roof,
                "cpu_baseline": cpu}
        print(json.dumps(line), flush=True)
    _finish(world, (graph,))


def run_rollout(args, wl, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import dlwp_benchmark_b200 as pkg
    from dlwp_benchmark_b200 import _lib
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = build_model(wl).to(dev).eval()
    B, R = wl["batch"], wl["rollout_steps"]
    g = torch.Generator().manual_seed(1234 + rank)
    hx = torch.randn(B, wl["cin"], wl["H"], wl["W"], generator=g).pin_memory()
    x0 = hx.to(dev)
    out = torch.empty(B, R, wl["cout"], wl["H"], wl["W"], device=dev)
    hlast = torch.empty(B, wl["cout"], wl["H"], wl["W"]).pin_memory()
    eng = pkg.Rollout(model, graph=not args.no_graph)
    lib = _lib.load()
    eng(x0, 2)                                                    # capture + first replay
    torch.cuda.synchronize()
    n0 = lib.sb200_kernel_launches()
    pkg.Rollout(model, graph=False)(x0, 1)
    torch.cuda.synchronize()
    launches = int(lib.sb200_kernel_launches() - n0)            # library kernels per model step
    t_dev, clocks = _timed(lambda: eng(x0, R, out), args.steps, args.warmup, world, local_rank, dist)

    def step_e2e():
        x0.copy_(hx, non_blocking=True)
        eng(x0, R, out)
        hlast.copy_(out[:, -1], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t_e2e, _ = _timed(step_e2e, args.steps, 1, world, local_rank, dist)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"output": out})          # [B, R, C, H, W] frames of the last rollout
    tt = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = tt.tolist()
    if rank == 0:
        peak, peak_src = _peak()
        C, L = wl["hidden"], wl["L"]
        P = B * C * wl["H"] * wl["W"]
        M = wl["n_modes"][0] * (wl["n_modes"][1] // 2 + 1)
        alg = L * (8 * P + 8 * C * C * M + 4 * C * C) + 2 * 4 * P          # SURVEY 8(d) fwd bytes per layer + lifting out / projection in
        per_model_step = t_dev / args.steps / R
        line = {"metric": "FNO2D closed-loop rollout IC-steps/s", "value": B * world * R * args.steps / t_dev,
                "unit": "IC-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": t_dev / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": wl["desc"], "global_ics": B * world, "rollout_steps": R, "grid": [wl["H"], wl["W"]],
                           "parallelism": f"ic-shard x{world} (no collective)", "step": "one 100-step closed-loop rollout",
                           "cuda_graph": not args.no_graph, "ms_per_model_step": per_model_step * 1e3,
                           "l2": "one activation tensor is 2.1 GB, far beyond the 126 MB L2"},
                "clocks": clocks,
                "e2e": {"value": B * world * R * args.steps / t_e2e, "unit": "IC-steps/s",
                        "h2d_bytes_per_step": hx.numel() * 4 * world, "d2h_bytes_per_step": hlast.numel() * 4 * world,
                        "ms_per_step": t_e2e / args.steps * 1e3, "note": "initial conditions H2D, last frame D2H per rollout"},
                "gpu_launches": launches * R * args.steps,
                "roofline": {"bound": "hbm", "kernel": "one model step (all kernels, forward only)",
                             "achieved": alg / per_model_step / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg / per_model_step / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "alg_bytes": alg},
                "cpu_baseline": cpu_rollout_rate(wl) if (world == 1 and not args.skip_cpu) else None}
        print(json.dumps(line), flush=True)
    _finish(world, (getattr(eng, "_graph", None),))


# ----------------------------------------------------------------------------------------
# the B200 arm
# ----------------------------------------------------------------------------------------
def run_b200(args, wl, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    import dlwp_benchmark_b200 as pkg  # noqa: F401  (fails loudly if the .so is missing)
    from dlwp_benchmark_b200.ddp import GradSync

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    model = build_model(wl).to(dev)
    params = [p for p in model.parameters()]
    opt = torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)
    sync = GradSync(params, world, avg=not args.ddp_sum) if world > 1 else None
    B = wl["batch"]
    g = torch.Generator().manual_seed(1234 + rank)
    hx = torch.randn(B, wl["cin"], wl["H"], wl["W"], generator=g).pin_memory()
    hy = torch.randn(B, wl["cout"], wl["H"], wl["W"], generator=g).pin_memory()
    x, y = hx.to(dev), hy.to(dev)
    loss_buf = torch.zeros((), device=dev)
    hloss = torch.zeros((), pin_memory=True)
    # output of the latest step (inside the graph: its static output), detached: holding its autograd graph would carry
    # the parameters' AccumulateGrad nodes of an eager step, bound to the eager stream, into the graph capture
    last = {}

    def fwd_bwd():
        out = model(x)
        last["out"] = out.detach()
        loss = torch.nn.functional.mse_loss(out, y)
        loss.backward()
        loss_buf.copy_(loss.detach())

    def step_eager():
        if sync:
            sync.zero()
        else:
            opt.zero_grad(set_to_none=True)
        fwd_bwd()
        if sync:
            sync.allreduce()
        opt.step()

    from dlwp_benchmark_b200 import _lib
    lib = _lib.load()
    if args.tc_mode is not None:
        _lib.set_tc_mode(args.tc_mode)
    step_eager()                                   # also the first-touch of plans / workspaces
    torch.cuda.synchronize()
    n0 = lib.sb200_kernel_launches()
    step_eager()
    torch.cuda.synchronize()
    launches_per_step = int(lib.sb200_kernel_launches() - n0)   # kernels of libspectral_b200.so per train step

    use_graph = not args.no_graph
    log(f'model built, graph={use_graph}, library kernel launches per step = {launches_per_step}')
    graph = None
    graph_mode = "whole step" if use_graph else "none"
    if use_graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                step_eager()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        if sync is None:
            opt.zero_grad(set_to_none=True)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                fwd_bwd()
                opt.step()
            step = graph.replay
        else:
            # grads live in GradSync's flat buffer (static addresses).  First choice: the whole step, NCCL
            # all-reduce and Adam included, as ONE graph; if this NCCL build refuses capture, keep the
            # collective and the optimizer outside the graph.
            step = None
            try:
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    sync.zero()
                    fwd_bwd()
                    sync.allreduce()
                    opt.step()
                torch.cuda.synchronize()
                graph.replay()
                torch.cuda.synchronize()
                step = graph.replay
                graph_mode = "whole step incl. NCCL all-reduce"
            except Exception as ex:  # noqa: BLE001
                log(f"whole-step capture failed ({ex!r}); capturing fwd+bwd only")
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    sync.zero()
                    fwd_bwd()
                graph_mode = "fwd+bwd (all-reduce + Adam eager)"

                def step():
                    graph.replay()
                    sync.allreduce()
                    opt.step()
    else:
        step = step_eager

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    log('step function ready')
    # ---- kernel-only (inputs resident) ----
    for _ in range(args.warmup):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as cs:
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    t_dev = e0.elapsed_time(e1) * 1e-3
    clocks = cs.summary()

    log(f'kernel-only timing done: {t_dev / args.steps * 1e3:.3f} ms/step')
    # ---- end to end: pinned host -> device every step, loss read back every step ----
    def step_e2e():
        x.copy_(hx, non_blocking=True)
        y.copy_(hy, non_blocking=True)
        step()
        hloss.copy_(loss_buf, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return float(hloss)

    for _ in range(min(args.warmup, 3)):
        step_e2e()
    barrier()
    e0.record()
    for _ in range(args.steps):
        last_loss = step_e2e()
    e1.record()
    barrier()
    t_e2e = e0.elapsed_time(e1) * 1e-3
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, _train_step_outputs(last["out"], loss_buf, model))

    tt = torch.tensor([t_dev, t_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_dev, t_e2e = tt.tolist()

    if rank == 0:
        peak, peak_src = _peak()
        roof = None
        log('e2e done; per-kernel rooflines')
        try:
            if args.skip_roofline:
                raise RuntimeError('skipped (--skip-roofline)')
            kr = kernel_rooflines(wl, peak)
            # launches per train step of each kernel on the spectral path (4 layers)
            L = wl["L"]
            per_step = {"analysis": 2 * L, "modes_gemm(mix_fwd)": 2 * L - 0,
                        "modes_gemm(wgrad)": L, "coldft_inv": 2 * L - 0, "rowidft_pointwise(fwd)": L,
                        "rowidft_pointwise(bwd)": L, "pointwise_wgrad": L}            # every other entry: once per step
            share = {k: v["ms"] * per_step.get(k, 1) for k, v in kr.items()}
            top = max(share, key=share.get)
            ncu_name = {"analysis": ("analysis_fused", None), "modes_gemm(mix_fwd)": ("modes_gemm2", None),
                        "modes_gemm(wgrad)": ("modes_gemm2", None), "coldft_inv": ("coldft_inv2", None),
                        "rowidft_pointwise(fwd)": ("tc_pointwise_kernel<3, 1, 0", None),
                        "rowidft_pointwise(bwd)": ("tc_pointwise_kernel<3, 3, 0", None),
                        "pointwise_wgrad": ("tc_wgrad_kernel<3, 0>", 8 * wl["batch"] * wl["hidden"] * wl["H"] * wl["W"])}
            ncu_name.update({"lift_fwd": ("tc_pointwise_kernel<3, 0, 1", None), "lift_wgrad": ("tc_wgrad_kernel<3, 1>", None),
                             "lift_tail_bwd": ("tc_pointwise_kernel<3, 7, 0", None),
                             "mlp_head_fwd": ("tc_pointwise_kernel<3, 5, 0", None),
                             "mlp_head_bwd(gz1 out)": ("tc_pointwise_kernel<3, 6, 0", None),
                             "head_dgrad(256->C)": ("tc_pointwise_kernel<3, 4, 0", None),
                             "head_wgrad(256xC)": ("tc_wgrad_kernel<3, 0>", 4 * wl["batch"] * (wl["proj"] + wl["hidden"]) * wl["H"] * wl["W"])})
            traffic = _ncu_traffic(*ncu_name[top]) if args.workload == "cfg2" and top in ncu_name else None
            roof = {"bound": "hbm", "kernel": top, "achieved": kr[top]["achieved_gbs"], "peak": peak,
                    "unit": "GB/s", "frac": kr[top]["frac"], "traffic": traffic,
                    "traffic_source": (_ncu_table_path(rel=True) + " (ncu --set full, same shapes)") if traffic else None,
                    "peak_source": peak_src,
                    "kernel_ms": kr[top]["ms"], "alg_bytes": kr[top]["alg_bytes"],
                    "all": {k: {"ms": round(v["ms"], 4), "frac": round(v["frac"], 4)} for k, v in kr.items()}}
        except Exception as ex:  # the roofline block must never take the headline number down
            roof = {"bound": "hbm", "error": repr(ex)}
        cpu = None
        gpu_cmp = None
        if world == 1 and not args.skip_cpu:
            log('gpu torch.fft comparison')
            gpu_cmp = gpu_torch_rate(wl, B)
            log('cpu baseline')
            sample = _cpu_sample(wl)
            rate, med, cores = cpu_oracle_rate(wl, sample, 10, 2)
            cpu = {"value": rate, "unit": "samples/s", "cores": cores, "kind": "port",
                   "sample": f"batch {sample} of {B}, fwd+MSE+bwd+Adam, 10 steps after 2 warm-up "
                             f"({12 * med:.1f} s of CPU work), oracle restatement"}
        n_launch = launches_per_step
        line = {
            "metric": "FNO2D train samples/s (fwd+bwd)", "value": B * world * args.steps / t_dev, "unit": "samples/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": _config(wl, world),
            "run": {"cuda_graph": bool(use_graph), "graph_scope": graph_mode, "tc_mode": int(_lib.tc_mode()),
                    "optimizer": "Adam(fused, capturable)", "grad_sync": "GradSync(direct sinks, 1 AVG all-reduce)" if sync else None},
            "clocks": clocks,
            "e2e": {"value": B * world * args.steps / t_e2e, "unit": "samples/s",
                    "h2d_bytes_per_step": (hx.numel() + hy.numel()) * 4 * world, "d2h_bytes_per_step": 4 * world,
                    "ms_per_step": t_e2e / args.steps * 1e3, "last_loss": last_loss},
            "gpu_launches": n_launch * args.steps,
            "roofline": roof,
            "cpu_baseline": cpu,
            "gpu_torch_baseline": gpu_cmp,
        }
        print(json.dumps(line), flush=True)
    _finish(world, (graph,))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default: 200 (b200 arm), 20 (reference arm)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--tc-mode", type=int, default=int(os.environ["SB200_TC_MODE"]) if os.environ.get("SB200_TC_MODE") else None,
                    help="0 = CUDA-core fp32, 1 = single-pass TF32 (parity ~1e-3), 3 = 3xTF32 (parity <= 1e-5; library default)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--ddp-sum", action="store_true", help="gradient all-reduce as SUM + scale instead of ReduceOp.AVG")
    ap.add_argument("--skip-roofline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last step as DIR/<name>.npy (b200 arm)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)
    if args.steps is None:
        args.steps = 20 if (args.impl == "reference" or args.workload in ("cfg3", "cfg5")) else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        if wl.get("kind"):
            if rank == 0:
                print(json.dumps({"impl": "reference", "unavailable": "the reference arm covers the FNO train-step workloads"}))
            return
        run_reference(args, wl, rank, world)
        return
    if wl.get("kind") in ("afno", "afnonet"):
        run_afno(args, wl, rank, world, local_rank)
    elif wl.get("kind") == "rollout":
        run_rollout(args, wl, rank, world, local_rank)
    else:
        run_b200(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
